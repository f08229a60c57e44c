// libsso_b200.so — the C ABI declared in include/sso_b200.h.
//
// Everything the operator's `contribute` / `verify_transcript` binaries reach through
// phase1_cli / phase2_cli on this path (SURVEY.md §8) is computed on the GPU; the host side
// only moves bytes, hashes (Blake2b, sequential by construction) and checks sizes.
// There is no CPU fallback: without a device every compute entry returns SSO_E_CUDA.
#include "flows.cuh"
#include "files.cuh"
#include "p2.cuh"
#include "p2prep.cuh"
#include <memory>
#include <thread>
#include <mutex>
#include <atomic>

using namespace sso;

// ---------------------------------------------------------------------------------------------
// small kernels that are not per-curve
// ---------------------------------------------------------------------------------------------
template <class F>
__global__ void k_test_field_mul(const uint8_t* a, const uint8_t* b, uint8_t* out, uint32_t n, uint32_t* status) {
  uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= n) return;
  typename F::T x, y;
  uint32_t fl;
  bool ok = F::from_bytes(a + (size_t)tid * F::NBYTES, false, fl, x);
  ok = F::from_bytes(b + (size_t)tid * F::NBYTES, false, fl, y) && ok;
  if (!ok) report(status, ST_NONCANONICAL, tid);
  F::to_bytes(out + (size_t)tid * F::NBYTES, F::mul(x, y), 0);
}

// Multiply-accumulate peak probes (roofline denominator, SURVEY.md §8d).
//   variant 0: mad.wide.u32 (32x32+64 -> 64) on 8 independent accumulators per thread
//   variant 1: the mad.lo.cc / madc.hi.cc carry-chain pairs the field multiplication is written in
//   variant 2: mad.lo.u32 (32x32+32 -> 32), for reference
// Every variant issues 32 multiply-accumulates per thread per iteration.
__global__ void k_imad_probe(uint32_t iters, uint32_t variant, uint32_t seed, uint64_t* sink) {
  uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t a = seed * 2654435761u + tid, b = (seed ^ 0x9e3779b9u) + tid * 7u;
  if (variant == 0) {
    uint64_t acc[8];
#pragma unroll
    for (int i = 0; i < 8; i++) acc[i] = tid + i;
    for (uint32_t it = 0; it < iters; it++) {
#pragma unroll
      for (int u = 0; u < 4; u++) {
#pragma unroll
        for (int i = 0; i < 8; i++) asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc[i]) : "r"(a + i), "r"(b + u));
      }
    }
    uint64_t s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) s ^= acc[i];
    if (s == 0x1234567ull) sink[0] = s;
  } else if (variant == 1) {
    uint32_t acc[4][8];
#pragma unroll
    for (int c = 0; c < 4; c++)
#pragma unroll
      for (int i = 0; i < 8; i++) acc[c][i] = tid + i + c;
    for (uint32_t it = 0; it < iters; it++) {
#pragma unroll
      for (int u = 0; u < 2; u++) {
#pragma unroll
        for (int c = 0; c < 4; c++) {
          // one carry chain of 4 products (8 half-instructions) per accumulator row
          acc[c][0] = mad_lo_cc(a + u, b + c, acc[c][0]);
          acc[c][1] = madc_hi_cc(a + u, b + c, acc[c][1]);
          acc[c][2] = madc_lo_cc(a + 1, b + c, acc[c][2]);
          acc[c][3] = madc_hi_cc(a + 1, b + c, acc[c][3]);
          acc[c][4] = madc_lo_cc(a + 2, b + c, acc[c][4]);
          acc[c][5] = madc_hi_cc(a + 2, b + c, acc[c][5]);
          acc[c][6] = madc_lo_cc(a + 3, b + c, acc[c][6]);
          acc[c][7] = madc_hi(a + 3, b + c, acc[c][7]);
        }
      }
    }
    uint32_t s = 0;
#pragma unroll
    for (int c = 0; c < 4; c++)
#pragma unroll
      for (int i = 0; i < 8; i++) s ^= acc[c][i];
    if (s == 0x1234567u) sink[0] = s;
  } else {
    uint32_t acc[8];
#pragma unroll
    for (int i = 0; i < 8; i++) acc[i] = tid + i;
    for (uint32_t it = 0; it < iters; it++) {
#pragma unroll
      for (int u = 0; u < 4; u++) {
#pragma unroll
        for (int i = 0; i < 8; i++) asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+r"(acc[i]) : "r"(a + i), "r"(b + u));
      }
    }
    uint32_t s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) s ^= acc[i];
    if (s == 0x1234567u) sink[0] = s;
  }
}

namespace sso {
ProfSlot g_prof[PK_COUNT];
std::atomic<int> g_prof_enabled{0};

// field_probe.cu (test-only kernels of sso_test_field_op)
int run_field_op(Ctx& c, int si, uint32_t field, const uint32_t* d_ops, const uint32_t* d_a, const uint32_t* d_b, const uint32_t* d_k,
                 uint32_t* d_out, uint32_t* d_rc, uint64_t n, char* err, size_t errcap);
}  // namespace sso

namespace {

const CurveOps* ops_for(uint32_t curve) {
  switch (curve) {
    case SSO_CURVE_BLS12_377: return curve_ops_bls12_377();
    case SSO_CURVE_BW6_761: return curve_ops_bw6_761();
    case SSO_CURVE_MNT4_753: return curve_ops_mnt4_753();
    case SSO_CURVE_MNT6_753: return curve_ops_mnt6_753();
  }
  return nullptr;
}

// n is bounded by the callers: vectors longer than 2^24 elements go through the piece engine (stream.cuh)
inline VecSeg seg(const uint8_t* in, uint8_t* out, uint64_t n, uint32_t slot, uint32_t has_coeff, uint32_t mode) {
  VecSeg s;
  s.in = in; s.out = out; s.n = n > 0xffffffffull ? 0xffffffffu : (uint32_t)n; s.coeff_slot = slot; s.has_coeff = has_coeff; s.mode = mode;
  return s;
}
inline VecBatch batch_of(std::initializer_list<VecSeg> segs) {
  VecBatch b;
  memset(&b, 0, sizeof b);
  for (const VecSeg& s : segs) {
    if (s.n == 0) continue;
    b.seg[b.nseg++] = s;
    b.total += s.n;
  }
  return b;
}

// Phase1::computation on the five vectors of one chunk: ONE tau-table launch, ONE batch_exp launch and ONE
// normalisation launch covering the three G1 vectors and tauG2 + betaG2.  Coefficient slots: 0 = 1, 1 = alpha, 2 = beta.
int p1_contribute_streams(Ctx& c, const CurveOps* ops, const P1Layout& L, const uint8_t* d_ch, uint8_t* d_resp,
                          const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta, uint32_t check, uint32_t* d_status,
                          char* err, size_t errcap) {
  int rc;
  const uint8_t* coeffs[TAU_COEFF_SLOTS] = {nullptr, alpha, beta};
  uint32_t* d_table;
  if (check == CHECK_FULL) {
    // CheckForCorrectness::Full on the inputs (--force-correctness-checks, reference src/bin/contribute.rs:816-819): on
    // the curve AND in the prime-order subgroup — a separate pass, so that the hot kernel keeps its register budget
    const uint64_t counts[5] = {L.g1n, L.on, L.on, L.on, 1};
    static const uint32_t groups[5] = {GROUP_G1, GROUP_G2, GROUP_G1, GROUP_G1, GROUP_G2};
    for (int v = 0; v < 5; v++)
      if (counts[v] && (rc = ops->reencode(c, 0, groups[v], d_ch + L.off_u[v], 0, counts[v], nullptr, 0, CHECK_FULL, 1, nullptr, d_status, err, errcap))) return rc;
  }
  if ((rc = ops->tau_tables(c, 0, L.start, tau, coeffs, &d_table, err, errcap))) return rc;
  VecBatch g2 = batch_of({seg(d_ch + L.off_u[1], d_resp + L.off_c[1], L.on, 0, 0, 0),
                          seg(d_ch + L.off_u[4], d_resp + L.off_c[4], 1, 2, 1, 1)});
  VecBatch g1 = batch_of({seg(d_ch + L.off_u[0], d_resp + L.off_c[0], L.g1n, 0, 0, 0),
                          seg(d_ch + L.off_u[2], d_resp + L.off_c[2], L.on, 1, 1, 0),
                          seg(d_ch + L.off_u[3], d_resp + L.off_c[3], L.on, 2, 1, 0)});
  // one launch for both groups: G2 blocks (longest-running) first, G1 blocks fill the tail
  return ops->batch_exp_chunk(c, 0, g1, g2, 0, d_table, 1, check, d_status, err, errcap);
}

// one vector, one scalar rule
int single_vector(Ctx& c, const CurveOps* ops, uint32_t group, const uint8_t* d_in, uint32_t in_compressed, uint64_t n,
                  uint64_t first_index, const uint8_t* tau, const uint8_t* coeff, uint32_t mode, uint8_t* d_out,
                  uint32_t out_compressed, uint32_t check, uint32_t* d_status, char* err, size_t errcap) {
  int rc;
  const uint8_t* coeffs[TAU_COEFF_SLOTS] = {coeff, nullptr, nullptr};
  uint32_t* d_table;
  if ((rc = ops->tau_tables(c, 0, first_index, tau, coeffs, &d_table, err, errcap))) return rc;
  VecBatch b = batch_of({seg(d_in, d_out, n, 0, coeff != nullptr, mode)});
  return ops->batch_exp(c, 0, group, b, in_compressed, d_table, out_compressed, check, d_status, err, errcap);
}

// one vector of points on the device and the checks it is decoded with
struct PairInput { const uint8_t* d; uint32_t compressed, check, subgroup; };

// Decodes n points to affine and returns on the host the random-linear-combination pair (two uncompressed points):
// (sum r_i a_i, sum r_i a_{i+1}) over n - 1 terms [power_pairs] when b.d is null, else (sum r_i a_i, sum r_i b_i) [merge_pairs].
// A point that fails its check is reported as `what`.
int pair_to_host(Ctx& c, const CurveOps* ops, uint32_t group, size_t usz, uint64_t n, PairInput a, PairInput b, const uint8_t* seed32,
                 const uint64_t* tweak, uint32_t* d_status, const char* what, uint8_t* pair, char* err, size_t errcap) {
  int rc;
  const size_t aff = ops->aff_words[group];
  uint32_t *d_aff_a, *d_aff_b = nullptr;
  uint8_t* d_pair;
  if ((rc = c.alloc((void**)&d_aff_a, n * aff * 4))) return rc;
  if (b.d && (rc = c.alloc((void**)&d_aff_b, n * aff * 4))) return rc;
  if ((rc = c.alloc((void**)&d_pair, 2 * usz))) return rc;
  if ((rc = ops->reencode(c, 0, group, a.d, a.compressed, n, nullptr, 0, a.check, a.subgroup, d_aff_a, d_status, err, errcap))) return rc;
  if (b.d && (rc = ops->reencode(c, 0, group, b.d, b.compressed, n, nullptr, 0, b.check, b.subgroup, d_aff_b, d_status, err, errcap))) return rc;
  if ((rc = ops->msm_pairs(c, 0, group, d_aff_a, b.d ? d_aff_b : d_aff_a + aff, b.d ? n : n - 1, seed32, tweak, d_pair, err, errcap))) return rc;
  if ((rc = sync_all(c, err, errcap))) return rc;
  if ((rc = check_status(c, d_status, what, err, errcap))) return rc;
  CUDA_TRY(cudaMemcpy(pair, d_pair, 2 * usz, cudaMemcpyDeviceToHost));
  return SSO_OK;
}

// batch_exp (mode 0: tau^(first_index + i) [* coeff]) and batch_mul (mode 1: the index-independent scalar `coeff`) of one vector.
// Vectors longer than the span of one tau table (2^24 indices) are processed in segments, each with its own table base.
int32_t batch_scalar_dev(uint32_t curve, uint32_t group, const void* d_in, uint32_t in_compressed, uint64_t n, uint64_t first_index,
                         const uint8_t* tau, const uint8_t* coeff, uint32_t mode, void* d_out, uint32_t out_compressed, uint32_t check_input,
                         int device, char* err, size_t errcap) {
  const CurveOps* ops = ops_for(curve);
  if (!ops || !(mode ? coeff : tau)) { set_err(err, errcap, "unknown curve %u or null scalar", curve); return SSO_E_ARG; }
  Ctx c(err, errcap);
  int rc = c.init(device);
  if (rc) return rc;
  uint32_t* d_status;
  if ((rc = status_buffer(c, &d_status, 0, true, err, errcap))) return rc;
  if (group > 1) { set_err(err, errcap, "unknown group %u", group); return SSO_E_ARG; }
  std::vector<uint8_t> one(ops->fr_bytes, 0);
  one[0] = 1;
  CurveSizes cs;
  curve_sizes(curve, cs);
  const uint64_t in_sz = point_size(cs, group, in_compressed), out_sz = point_size(cs, group, out_compressed);
  const uint64_t SEG = 1ull << 22;
  for (uint64_t off = 0; off < n; off += SEG) {
    uint64_t m = n - off < SEG ? n - off : SEG;
    if ((rc = single_vector(c, ops, group, (const uint8_t*)d_in + off * in_sz, in_compressed, m, mode ? 0 : first_index + off,
                            mode ? one.data() : tau, coeff, mode, (uint8_t*)d_out + off * out_sz, out_compressed, check_input, d_status,
                            err, errcap))) return rc;
  }
  if ((rc = sync_all(c, err, errcap))) return rc;
  return check_status(c, d_status, mode ? "batch_mul input" : "batch_exp input", err, errcap);
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

const char* sso_version(void) { return "sso_b200 0.1 (sm_100a)"; }

int32_t sso_device_count(void) {
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess) return 0;
  return cnt;
}

int32_t sso_device_name(int device, char* out, size_t cap) {
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return SSO_E_CUDA;
  snprintf(out, cap, "%s", prop.name);
  return SSO_OK;
}

int32_t sso_curve_sizes(uint32_t curve, uint64_t out[5]) {
  CurveSizes s;
  if (!curve_sizes(curve, s)) return SSO_E_ARG;
  out[0] = s.g1c; out[1] = s.g1u; out[2] = s.g2c; out[3] = s.g2u; out[4] = s.fr;
  return SSO_OK;
}

int32_t sso_p1_sizes(const sso_p1_params_t* p, uint64_t out[8], char* err, size_t errcap) {
  P1Layout L;
  int rc = p1_layout(p, L, err, errcap);
  if (rc) return rc;
  out[SSO_SZ_POWERS_LENGTH] = L.powers_length;
  out[SSO_SZ_POWERS_G1_LENGTH] = L.powers_g1_length;
  out[SSO_SZ_G1_COUNT] = L.g1n;
  out[SSO_SZ_OTHER_COUNT] = L.on;
  out[SSO_SZ_ACCUMULATOR] = L.acc_size;
  out[SSO_SZ_CONTRIBUTION] = L.contrib_size;
  out[SSO_SZ_PUBLIC_KEY] = L.pk_size;
  out[SSO_SZ_NUM_CHUNKS] = L.num_chunks;
  return SSO_OK;
}

int32_t sso_blake2b_512(const uint8_t* data, size_t len, uint8_t out[64]) {
  blake2b_512(data, len, out);
  return SSO_OK;
}

int32_t sso_batch_exp_dev(uint32_t curve, uint32_t group, const void* d_in, uint32_t in_compressed, uint64_t n,
                          uint64_t first_index, const uint8_t* tau, const uint8_t* coeff, void* d_out,
                          uint32_t out_compressed, uint32_t check_input, int device, char* err, size_t errcap) {
  return batch_scalar_dev(curve, group, d_in, in_compressed, n, first_index, tau, coeff, 0, d_out, out_compressed, check_input, device, err, errcap);
}

int32_t sso_batch_mul_dev(uint32_t curve, uint32_t group, const void* d_in, uint32_t in_compressed, uint64_t n,
                          const uint8_t* scalar, void* d_out, uint32_t out_compressed, uint32_t check_input,
                          int device, char* err, size_t errcap) {
  return batch_scalar_dev(curve, group, d_in, in_compressed, n, 0, nullptr, scalar, 1, d_out, out_compressed, check_input, device, err, errcap);
}

int32_t sso_reencode_dev(uint32_t curve, uint32_t group, const void* d_in, uint32_t in_compressed, uint64_t n,
                         void* d_out, uint32_t out_compressed, uint32_t check, uint32_t subgroup_check,
                         int device, char* err, size_t errcap) {
  const CurveOps* ops = ops_for(curve);
  if (!ops) { set_err(err, errcap, "unknown curve %u", curve); return SSO_E_ARG; }
  Ctx c(err, errcap);
  int rc = c.init(device);
  if (rc) return rc;
  uint32_t* d_status;
  if ((rc = status_buffer(c, &d_status, 0, true, err, errcap))) return rc;
  if ((rc = ops->reencode(c, 0, group, (const uint8_t*)d_in, in_compressed, n, (uint8_t*)d_out, out_compressed, check,
                          subgroup_check, nullptr, d_status, err, errcap))) return rc;
  if ((rc = sync_all(c, err, errcap))) return rc;
  return check_status(c, d_status, "point", err, errcap);
}

// K3 + K5: validate/decode n points and return (sum r_i v_i, sum r_i v_{i+1}) [power_pairs] as two uncompressed points
int32_t sso_power_pairs_dev(uint32_t curve, uint32_t group, const void* d_in, uint32_t in_compressed, uint64_t n,
                            uint32_t check, uint32_t subgroup_check, const uint8_t* seed32, uint8_t* out_pair, size_t out_len,
                            int device, char* err, size_t errcap) {
  const CurveOps* ops = ops_for(curve);
  if (!ops || group > 1) { set_err(err, errcap, "unknown curve/group %u/%u", curve, group); return SSO_E_ARG; }
  if (n < 2) { set_err(err, errcap, "power_pairs needs at least two elements"); return SSO_E_ARG; }
  CurveSizes cs;
  curve_sizes(curve, cs);
  const size_t usz = point_size(cs, group, 0);
  if (out_len != 2 * usz) { set_err(err, errcap, "output buffer must hold two uncompressed points (%llu bytes)", (unsigned long long)(2 * usz)); return SSO_E_ARG; }
  Ctx c(err, errcap);
  int rc = c.init(device);
  if (rc) return rc;
  uint32_t* d_status;
  if ((rc = status_buffer(c, &d_status, 0, true, err, errcap))) return rc;
  return pair_to_host(c, ops, group, usz, n, {(const uint8_t*)d_in, in_compressed, check, subgroup_check}, {}, seed32, nullptr, d_status,
                      "point", out_pair, err, errcap);
}

// K3 + K5: (sum r_i a_i, sum r_i b_i) [merge_pairs] for two vectors of n points each
int32_t sso_merge_pairs_dev(uint32_t curve, uint32_t group, const void* d_a, const void* d_b, uint32_t in_compressed, uint64_t n,
                            uint32_t check, uint32_t subgroup_check, const uint8_t* seed32, uint8_t* out_pair, size_t out_len,
                            int device, char* err, size_t errcap) {
  const CurveOps* ops = ops_for(curve);
  if (!ops || group > 1) { set_err(err, errcap, "unknown curve/group %u/%u", curve, group); return SSO_E_ARG; }
  if (n < 1) { set_err(err, errcap, "merge_pairs needs at least one element"); return SSO_E_ARG; }
  CurveSizes cs;
  curve_sizes(curve, cs);
  const size_t usz = point_size(cs, group, 0);
  if (out_len != 2 * usz) { set_err(err, errcap, "output buffer must hold two uncompressed points (%llu bytes)", (unsigned long long)(2 * usz)); return SSO_E_ARG; }
  Ctx c(err, errcap);
  int rc = c.init(device);
  if (rc) return rc;
  uint32_t* d_status;
  if ((rc = status_buffer(c, &d_status, 0, true, err, errcap))) return rc;
  return pair_to_host(c, ops, group, usz, n, {(const uint8_t*)d_a, in_compressed, check, subgroup_check},
                      {(const uint8_t*)d_b, in_compressed, check, subgroup_check}, seed32, nullptr, d_status, "point", out_pair, err, errcap);
}

// K8: batch of same_ratio checks on host buffers
int32_t sso_same_ratio(uint32_t curve, const uint8_t* checks, uint64_t n, uint32_t* verdicts, int device, char* err,
                       size_t errcap) {
  const CurveOps* ops = ops_for(curve);
  if (!ops || !checks || !verdicts) { set_err(err, errcap, "unknown curve %u or null buffer", curve); return SSO_E_ARG; }
  if (n == 0) return SSO_OK;
  Ctx c(err, errcap);
  int rc = c.init(device);
  if (rc) return rc;
  uint8_t* d_checks;
  uint32_t* d_verdicts;
  if ((rc = c.alloc((void**)&d_checks, n * ops->check_bytes))) return rc;
  if ((rc = c.alloc((void**)&d_verdicts, n * 4))) return rc;
  CUDA_TRY(cudaMemcpyAsync(d_checks, checks, n * ops->check_bytes, cudaMemcpyHostToDevice, c.s[0]));
  if ((rc = ops->same_ratio(c, 0, d_checks, n, d_verdicts, err, errcap))) return rc;
  if ((rc = sync_all(c, err, errcap))) return rc;
  CUDA_TRY(cudaMemcpy(verdicts, d_verdicts, n * 4, cudaMemcpyDeviceToHost));
  for (uint64_t i = 0; i < n; i++)
    if (verdicts[i] >= 0x100u) {
      set_err(err, errcap, "same_ratio check %llu: %s", (unsigned long long)i, status_text(verdicts[i] - 0x100u));
      return SSO_E_INPUT;
    }
  return SSO_OK;
}

int32_t sso_p1_contribute_dev(const sso_p1_params_t* p, const void* d_challenge, void* d_response,
                              const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta,
                              uint32_t check_input, int device, char* err, size_t errcap) {
  P1Layout L;
  int rc = p1_layout(p, L, err, errcap);
  if (rc) return rc;
  const CurveOps* ops = ops_for(p->curve);
  if (!tau || !alpha || !beta) { set_err(err, errcap, "null scalar"); return SSO_E_ARG; }
  Ctx c(err, errcap);
  if ((rc = c.init(device, 2))) return rc;
  uint32_t* d_status;
  if ((rc = status_buffer(c, &d_status, 0, true, err, errcap))) return rc;
  if ((rc = p1_contribute_streams(c, ops, L, (const uint8_t*)d_challenge, (uint8_t*)d_response, tau, alpha, beta, check_input, d_status, err, errcap))) return rc;
  if ((rc = sync_all(c, err, errcap))) return rc;
  return check_status(c, d_status, "challenge", err, errcap);
}

// Full-mode accumulators and chunks beyond what one launch set should hold are streamed in pieces (stream.cuh)
static bool needs_streaming(const sso_p1_params_t* p, const P1Layout& L) {
  // Full mode is the whole-accumulator case (beacon contribution and its verification): always in `batch_size` pieces
  const uint64_t big = 1ull << 22;
  return L.g1n > big || L.on > big || p->contribution_mode == SSO_MODE_FULL;
}

// phase1_cli::contribute on an accumulator streamed in `batch_size` pieces over the participants (devices of this process or
// the ranks of the process group): the beacon contribution on the combined file (reference src/bin/verify_transcript.rs:675-696,
// src/bin/control.rs:792-808).  With a process group every rank computes its own pieces into the shared response mapping;
// the hash and the proofs of knowledge are computed redundantly (identical bytes).
static int32_t contribute_streamed(const sso_p1_params_t* p, const P1Layout& L, const CurveOps* ops, const uint8_t* challenge, uint8_t* response,
                                   const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta, const uint8_t* pubkey, const uint8_t* seed32,
                                   uint32_t check_input, int device, char* err, size_t errcap) {
  int rc;
  Participants P;
  if ((rc = resolve_participants(nullptr, 0, device, p->contribution_mode == SSO_MODE_FULL, P, err, errcap))) return rc;
  std::thread hasher([=] { blake2b_512(challenge, L.acc_size, response); });
  JoinOnExit join_hasher{hasher};
  Ctx c(err, errcap);
  if ((rc = c.init(P.devices[0], 1))) return rc;
  std::vector<uint8_t> scalars;
  KeygenState keys;
  if (seed32) {
    scalars.resize(3 * (size_t)L.cs.fr);
    if ((rc = keygen_stage1(c, 0, ops, L.cs, seed32, 3, keys, scalars.data(), err, errcap))) return rc;
    tau = scalars.data(); alpha = scalars.data() + L.cs.fr; beta = scalars.data() + 2 * (size_t)L.cs.fr;
  }
  if ((rc = stream_contribute(ops, L, challenge, response, tau, alpha, beta, check_input, p->batch_size, P, err, errcap))) return rc;
  hasher.join();
  if (seed32) {
    if ((rc = keygen_stage2(c, 0, ops, L.cs, response, keys, response + L.off_c[5], err, errcap))) return rc;
    CUDA_TRY(cudaStreamSynchronize(c.s[0]));
  } else if (pubkey) memcpy(response + L.off_c[5], pubkey, L.pk_size);
  return SSO_OK;
}

// Shared body of sso_p1_contribute_buf (scalars and public key given) and sso_p1_contribute_seeded_buf (seed32 given:
// scalars drawn first, proofs of knowledge computed once the challenge hash is known, on a high-priority stream beside
// the main kernels).  The challenge is hashed ONCE, on the host, while the GPU works.
static int32_t contribute_buf_core(const sso_p1_params_t* p, const uint8_t* challenge, size_t challenge_len, uint8_t* response,
                                   size_t response_len, const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta,
                                   const uint8_t* pubkey, size_t pubkey_len, const uint8_t* seed32, uint32_t check_input, int device,
                                   char* err, size_t errcap) {
  P1Layout L;
  int rc = p1_layout(p, L, err, errcap);
  if (rc) return rc;
  const CurveOps* ops = ops_for(p->curve);
  if (!challenge || !response || (!seed32 && (!tau || !alpha || !beta))) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  if (challenge_len != L.acc_size) { set_err(err, errcap, "challenge has %zu bytes, expected accumulator_size %llu", challenge_len, (unsigned long long)L.acc_size); return SSO_E_ARG; }
  if (response_len != L.contrib_size) { set_err(err, errcap, "response has %zu bytes, expected contribution_size %llu", response_len, (unsigned long long)L.contrib_size); return SSO_E_ARG; }
  if (pubkey && pubkey_len != L.pk_size) { set_err(err, errcap, "public key has %zu bytes, expected %llu", pubkey_len, (unsigned long long)L.pk_size); return SSO_E_ARG; }
  if (needs_streaming(p, L)) return contribute_streamed(p, L, ops, challenge, response, tau, alpha, beta, pubkey, seed32, check_input, device, err, errcap);
  Ctx c(err, errcap);
  if ((rc = c.init(device, seed32 ? 3 : 2))) return rc;
  std::vector<uint8_t> scalars;
  KeygenState keys;
  // the hash-chain link is computed on the host while the GPU works; with a seed it starts before the key generation
  // (whose first stage is a ~19 ms single-thread kernel the host would otherwise wait for)
  std::thread hasher;
  JoinOnExit join_hasher{hasher};
  if (seed32) {
    hasher = std::thread([=] { blake2b_512(challenge, challenge_len, response); });
    scalars.resize(3 * (size_t)L.cs.fr);
    if ((rc = keygen_stage1(c, 2, ops, L.cs, seed32, 3, keys, scalars.data(), err, errcap))) return rc;   // high-priority stream: not queued behind other chunks' kernels
    tau = scalars.data();
    alpha = scalars.data() + L.cs.fr;
    beta = scalars.data() + 2 * (size_t)L.cs.fr;
    c.mark("keygen: scalars");
  }
  uint8_t *d_ch, *d_resp;
  uint32_t* d_status;
  if ((rc = c.alloc((void**)&d_ch, L.acc_size))) return rc;
  if ((rc = c.alloc((void**)&d_resp, L.contrib_size))) return rc;
  if ((rc = status_buffer(c, &d_status, 0, true, err, errcap))) return rc;
  c.mark("scratch allocated");
  // stream-ordered: the kernels below are enqueued behind the copy, and the host goes straight on to hashing
  CUDA_TRY(cudaMemcpyAsync(d_ch, challenge, L.acc_size, cudaMemcpyHostToDevice, c.s[0]));
  c.mark("challenge H2D enqueued");
  if ((rc = p1_contribute_streams(c, ops, L, d_ch, d_resp, tau, alpha, beta, check_input, d_status, err, errcap))) return rc;
  c.mark("kernels enqueued");
  if (hasher.joinable()) hasher.join();
  else blake2b_512(challenge, challenge_len, response);
  c.mark("blake2b(challenge)");
  if (seed32) {
    if ((rc = keygen_stage2(c, 2, ops, L.cs, response, keys, response + L.off_c[5], err, errcap))) return rc;
    c.mark("keygen: proofs of knowledge enqueued");
  }
  if ((rc = sync_all(c, err, errcap))) return rc;
  if ((rc = check_status(c, d_status, "challenge", err, errcap))) return rc;
  CUDA_TRY(cudaMemcpy(response + 64, d_resp + 64, L.off_c[5] - 64, cudaMemcpyDeviceToHost));
  c.mark("response D2H");
  if (pubkey) memcpy(response + L.off_c[5], pubkey, L.pk_size);
  return SSO_OK;
}

int32_t sso_p1_contribute_buf(const sso_p1_params_t* p, const uint8_t* challenge, size_t challenge_len,
                              uint8_t* response, size_t response_len, const uint8_t* tau, const uint8_t* alpha,
                              const uint8_t* beta, const uint8_t* pubkey, size_t pubkey_len, uint32_t check_input,
                              int device, char* err, size_t errcap) {
  if (!tau || !alpha || !beta) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  return contribute_buf_core(p, challenge, challenge_len, response, response_len, tau, alpha, beta, pubkey, pubkey_len, nullptr,
                             check_input, device, err, errcap);
}

// Several chunks in flight (the reference runs up to --max-in-process-lane chunks through its Process lane,
// src/bin/contribute.rs:64-71, 158-163, 1132-1139; verify_transcript loops over the chunks of a round,
// src/bin/verify_transcript.rs:293-569): `host_threads` workers each take the next chunk and run the single-chunk
// call on their own streams, so the sequential Blake2b of one chunk overlaps the copies and kernels of the others and
// the throughput of the call is bound by the GPU, not by one host core.  device < 0: all visible devices, worker t on
// device t mod count (default 3 workers per device).
int32_t sso_p1_contribute_many_buf(const sso_p1_params_t* params, size_t n_chunks, const uint8_t* const* challenges,
                                   const size_t* challenge_lens, uint8_t* const* responses, const size_t* response_lens,
                                   const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta, const uint8_t* pubkey,
                                   size_t pubkey_len, uint32_t check_input, uint32_t host_threads, int device, char* err,
                                   size_t errcap) {
  if (!params || !challenges || !challenge_lens || !responses || !response_lens) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  return run_chunks_in_flight(n_chunks, host_threads, device, err, errcap, [&](size_t i, int dev, char* e, size_t ec) {
    return sso_p1_contribute_buf(&params[i], challenges[i], challenge_lens[i], responses[i], response_lens[i], tau, alpha, beta,
                                 pubkey, pubkey_len, check_input, dev, e, ec);
  });
}

int32_t sso_p1_new_challenge_dev(const sso_p1_params_t* p, void* d_challenge, int device, char* err, size_t errcap) {
  P1Layout L;
  int rc = p1_layout(p, L, err, errcap);
  if (rc) return rc;
  const CurveOps* ops = ops_for(p->curve);
  Ctx c(err, errcap);
  if ((rc = c.init(device, 2))) return rc;
  uint8_t* d = (uint8_t*)d_challenge;
  uint8_t blank[64];
  blake2b_512(nullptr, 0, blank);
  CUDA_TRY(cudaMemcpyAsync(d, blank, 64, cudaMemcpyHostToDevice, c.s[0]));
  if ((rc = ops->fill_generator(c, 0, GROUP_G1, L.g1n, d + L.off_u[0], 0, err, errcap))) return rc;
  if ((rc = ops->fill_generator(c, 1, GROUP_G2, L.on, d + L.off_u[1], 0, err, errcap))) return rc;
  if ((rc = ops->fill_generator(c, 0, GROUP_G1, 2 * L.on, d + L.off_u[2], 0, err, errcap))) return rc;
  if ((rc = ops->fill_generator(c, 1, GROUP_G2, 1, d + L.off_u[4], 0, err, errcap))) return rc;
  return sync_all(c, err, errcap);
}

int32_t sso_profile_enable(int32_t on) {
  g_prof_enabled.store(on == 2 ? 2 : (on ? 1 : 0));
  return SSO_OK;
}

int32_t sso_profile_reset(void) {
  for (auto& s : g_prof) { s.launches.store(0); s.ns.store(0); s.elems.store(0); }
  return SSO_OK;
}

int32_t sso_profile_read(uint64_t* out, size_t cap) {
  size_t need = (size_t)PK_COUNT * 3;
  if (cap < need) return SSO_E_ARG;
  for (int i = 0; i < PK_COUNT; i++) {
    out[3 * i] = g_prof[i].launches.load();
    out[3 * i + 1] = g_prof[i].ns.load();
    out[3 * i + 2] = g_prof[i].elems.load();
  }
  return (int32_t)PK_COUNT;
}

// Phase1::key_generation from the contributor seed (a3, a13)
int32_t sso_p1_keygen(uint32_t curve, const uint8_t seed32[32], const uint8_t digest64[64], uint8_t* scalars_out, size_t scalars_len,
                      uint8_t* pubkey_out, size_t pubkey_len, int device, char* err, size_t errcap) {
  const CurveOps* ops = ops_for(curve);
  CurveSizes cs;
  if (!ops || !curve_sizes(curve, cs) || !seed32 || !digest64) { set_err(err, errcap, "unknown curve %u or null argument", curve); return SSO_E_ARG; }
  if (scalars_len != 3 * cs.fr || pubkey_len != 6 * cs.g1u + 3 * cs.g2u) { set_err(err, errcap, "keygen: wrong output sizes"); return SSO_E_ARG; }
  Ctx c(err, errcap);
  int rc = c.init(device);
  if (rc) return rc;
  return keygen_host(c, ops, cs, seed32, digest64, 3, scalars_out, pubkey_out, err, errcap);
}

// phase1_cli::contribute on host buffers: hash, key generation from the seeded RNG, computation, public key
int32_t sso_p1_contribute_seeded_buf(const sso_p1_params_t* p, const uint8_t* challenge, size_t challenge_len, uint8_t* response,
                                     size_t response_len, const uint8_t seed32[32], uint32_t check_input, int device, char* err,
                                     size_t errcap) {
  if (!seed32) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  return contribute_buf_core(p, challenge, challenge_len, response, response_len, nullptr, nullptr, nullptr, nullptr, 0, seed32,
                             check_input, device, err, errcap);
}

// phase1_cli::contribute for several chunks in flight: the contributor applies the same seed-derived key to every
// chunk it holds (src/bin/contribute.rs:789, 809-823); worker / device semantics of sso_p1_contribute_many_buf
int32_t sso_p1_contribute_seeded_many_buf(const sso_p1_params_t* params, size_t n_chunks, const uint8_t* const* challenges,
                                          const size_t* challenge_lens, uint8_t* const* responses, const size_t* response_lens,
                                          const uint8_t seed32[32], uint32_t check_input, uint32_t host_threads, int device,
                                          char* err, size_t errcap) {
  if (!params || !challenges || !challenge_lens || !responses || !response_lens || !seed32) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  return run_chunks_in_flight(n_chunks, host_threads, device, err, errcap, [&](size_t i, int dev, char* e, size_t ec) {
    return sso_p1_contribute_seeded_buf(&params[i], challenges[i], challenge_lens[i], responses[i], response_lens[i], seed32,
                                        check_input, dev, e, ec);
  });
}

// Phase1::verification for one chunk on host buffers (a5)
static int32_t verify_chunk_core(const sso_p1_params_t* p, const uint8_t* challenge, size_t challenge_len, const uint8_t* response,
                                size_t response_len, uint8_t* new_challenge, size_t new_challenge_len, uint32_t check_input,
                                uint32_t check_output, uint32_t subgroup_check_mode, uint32_t ratio_check, const uint8_t* rlc_seed32,
                                int device, uint8_t* ch_hash_out, char* err, size_t errcap) {
  P1Layout L;
  int rc = p1_layout(p, L, err, errcap);
  if (rc) return rc;
  if (!challenge || !response || !new_challenge) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  if (challenge_len != L.acc_size || new_challenge_len != L.acc_size) { set_err(err, errcap, "challenge / new challenge must have accumulator_size %llu bytes", (unsigned long long)L.acc_size); return SSO_E_ARG; }
  if (response_len != L.contrib_size) { set_err(err, errcap, "response has %zu bytes, expected contribution_size %llu", response_len, (unsigned long long)L.contrib_size); return SSO_E_ARG; }
  const CurveOps* ops = ops_for(p->curve);
  uint64_t chunk_index = p->contribution_mode == SSO_MODE_FULL ? 0 : p->chunk_index;
  if (needs_streaming(p, L)) {
    Participants P;
    if ((rc = resolve_participants(nullptr, 0, device, p->contribution_mode == SSO_MODE_FULL, P, err, errcap))) return rc;
    Ctx c(err, errcap);
    if ((rc = c.init(P.devices[0], 1))) return rc;
    return verify_chunk_host(c, ops, L, p->curve, chunk_index, challenge, response, new_challenge, check_input, check_output,
                             subgroup_check_mode, ratio_check, rlc_seed32, &P, p->batch_size, ch_hash_out, err, errcap);
  }
  Ctx c(err, errcap);
  if ((rc = c.init(device, 2))) return rc;
  return verify_chunk_host(c, ops, L, p->curve, chunk_index, challenge, response, new_challenge, check_input, check_output,
                           subgroup_check_mode, ratio_check, rlc_seed32, nullptr, 0, ch_hash_out, err, errcap);
}

int32_t sso_p1_verify_chunk_buf(const sso_p1_params_t* p, const uint8_t* challenge, size_t challenge_len, const uint8_t* response,
                                size_t response_len, uint8_t* new_challenge, size_t new_challenge_len, uint32_t check_input,
                                uint32_t check_output, uint32_t subgroup_check_mode, uint32_t ratio_check, const uint8_t* rlc_seed32,
                                int device, char* err, size_t errcap) {
  return verify_chunk_core(p, challenge, challenge_len, response, response_len, new_challenge, new_challenge_len, check_input, check_output,
                           subgroup_check_mode, ratio_check, rlc_seed32, device, nullptr, err, errcap);
}

// The chunk loop of verify_transcript (src/bin/verify_transcript.rs:293-569) as a work queue: chunks are verified
// independently (the hash-chain order across rounds stays with the caller), several in flight per device.
int32_t sso_p1_verify_chunk_many_buf(const sso_p1_params_t* params, size_t n_chunks, const uint8_t* const* challenges,
                                     const size_t* challenge_lens, const uint8_t* const* responses, const size_t* response_lens,
                                     uint8_t* const* new_challenges, const size_t* new_challenge_lens, uint32_t check_input,
                                     uint32_t check_output, uint32_t subgroup_check_mode, uint32_t ratio_check,
                                     const uint8_t* rlc_seed32, uint32_t host_threads, int device, char* err, size_t errcap) {
  if (!params || !challenges || !challenge_lens || !responses || !response_lens || !new_challenges || !new_challenge_lens) {
    set_err(err, errcap, "null argument");
    return SSO_E_ARG;
  }
  return run_chunks_in_flight(n_chunks, host_threads, device, err, errcap, [&](size_t i, int dev, char* e, size_t ec) {
    return sso_p1_verify_chunk_buf(&params[i], challenges[i], challenge_lens[i], responses[i], response_lens[i], new_challenges[i],
                                   new_challenge_lens[i], check_input, check_output, subgroup_check_mode, ratio_check, rlc_seed32, dev, e, ec);
  });
}

// sum of n uncompressed points on host buffers (combining all-gathered per-GPU partial MSM results)
int32_t sso_points_sum(uint32_t curve, uint32_t group, const uint8_t* points, uint64_t n, uint8_t* out, size_t out_len, int device,
                       char* err, size_t errcap) {
  const CurveOps* ops = ops_for(curve);
  CurveSizes cs;
  if (!ops || group > 1 || !curve_sizes(curve, cs)) { set_err(err, errcap, "unknown curve/group %u/%u", curve, group); return SSO_E_ARG; }
  const size_t usz = point_size(cs, group, 0);
  if (out_len != usz || n == 0 || n > 65536) { set_err(err, errcap, "points_sum: bad sizes"); return SSO_E_ARG; }
  Ctx c(err, errcap);
  int rc = c.init(device);
  if (rc) return rc;
  uint8_t *d_in, *d_out;
  uint32_t* d_status;
  if ((rc = status_buffer(c, &d_status, 0, true, err, errcap))) return rc;
  if ((rc = c.alloc((void**)&d_in, n * usz))) return rc;
  if ((rc = c.alloc((void**)&d_out, usz))) return rc;
  CUDA_TRY(cudaMemcpyAsync(d_in, points, n * usz, cudaMemcpyHostToDevice, c.s[0]));
  if ((rc = ops->points_sum(c, 0, group, d_in, (uint32_t)n, d_out, d_status, err, errcap))) return rc;
  if ((rc = sync_all(c, err, errcap))) return rc;
  if ((rc = check_status(c, d_status, "point", err, errcap))) return rc;
  CUDA_TRY(cudaMemcpy(out, d_out, usz, cudaMemcpyDeviceToHost));
  return SSO_OK;
}

// phase-2 batch_mul of a G1 query vector (h_query / l_query) by delta^-1 on host buffers (a10 core)
int32_t sso_p2_scale_queries_buf(uint32_t curve, const uint8_t* in, size_t in_len, uint8_t* out, size_t out_len, uint64_t n,
                                 const uint8_t* delta_inv, uint32_t in_compressed, uint32_t out_compressed, uint32_t check_input,
                                 int device, char* err, size_t errcap) {
  CurveSizes cs;
  if (!curve_sizes(curve, cs) || !in || !out || !delta_inv) { set_err(err, errcap, "unknown curve %u or null argument", curve); return SSO_E_ARG; }
  const size_t isz = point_size(cs, GROUP_G1, in_compressed), osz = point_size(cs, GROUP_G1, out_compressed);
  if (in_len != n * isz || out_len != n * osz) { set_err(err, errcap, "query buffers have the wrong size for %llu points", (unsigned long long)n); return SSO_E_ARG; }
  if (n == 0) return SSO_OK;
  Ctx c(err, errcap);
  int rc = c.init(device);
  if (rc) return rc;
  uint8_t *d_in, *d_out;
  if ((rc = c.alloc((void**)&d_in, in_len))) return rc;
  if ((rc = c.alloc((void**)&d_out, out_len))) return rc;
  CUDA_TRY(cudaMemcpyAsync(d_in, in, in_len, cudaMemcpyHostToDevice, c.s[0]));
  CUDA_TRY(cudaStreamSynchronize(c.s[0]));
  if ((rc = sso_batch_mul_dev(curve, GROUP_G1, d_in, in_compressed, n, delta_inv, d_out, out_compressed, check_input, device, err, errcap))) return rc;
  CUDA_TRY(cudaMemcpy(out, d_out, out_len, cudaMemcpyDeviceToHost));
  return SSO_OK;
}

// phase-2 query check (a11 core): same_ratio(merge_pairs(before, after), (delta_g2_after, delta_g2_before))
int32_t sso_p2_verify_queries_buf(uint32_t curve, const uint8_t* before, size_t before_len, const uint8_t* after, size_t after_len,
                                  uint64_t n, uint32_t before_compressed, uint32_t after_compressed, const uint8_t* delta_g2_before,
                                  const uint8_t* delta_g2_after, uint32_t check, uint32_t subgroup_check, const uint8_t* rlc_seed32,
                                  int device, char* err, size_t errcap) {
  const CurveOps* ops = ops_for(curve);
  CurveSizes cs;
  if (!ops || !curve_sizes(curve, cs) || !before || !after || !delta_g2_before || !delta_g2_after) { set_err(err, errcap, "unknown curve %u or null argument", curve); return SSO_E_ARG; }
  const size_t bsz = point_size(cs, GROUP_G1, before_compressed), asz = point_size(cs, GROUP_G1, after_compressed);
  if (before_len != n * bsz || after_len != n * asz || n == 0) { set_err(err, errcap, "query buffers have the wrong size for %llu points", (unsigned long long)n); return SSO_E_ARG; }
  Ctx c(err, errcap);
  int rc = c.init(device);
  if (rc) return rc;
  uint8_t *d_b, *d_a;
  uint32_t* d_status;
  if ((rc = status_buffer(c, &d_status, 0, true, err, errcap))) return rc;
  if ((rc = c.alloc((void**)&d_b, before_len))) return rc;
  if ((rc = c.alloc((void**)&d_a, after_len))) return rc;
  CUDA_TRY(cudaMemcpyAsync(d_b, before, before_len, cudaMemcpyHostToDevice, c.s[0]));
  CUDA_TRY(cudaMemcpyAsync(d_a, after, after_len, cudaMemcpyHostToDevice, c.s[0]));
  const uint64_t tweak[4] = {TWEAK_P2_VERIFY, n, 0, 0};
  std::vector<uint8_t> pair(2 * cs.g1u);
  if ((rc = pair_to_host(c, ops, GROUP_G1, cs.g1u, n, {d_b, before_compressed, SSO_CHECK_NO, 0}, {d_a, after_compressed, check, subgroup_check},
                         rlc_seed32, tweak, d_status, "query", pair.data(), err, errcap))) return rc == SSO_E_INPUT ? SSO_E_VERIFY : rc;
  std::vector<RatioCheck> checks;
  add_check(checks, "phase-2 query vs delta_g2", pair.data(), pair.data() + cs.g1u, cs.g1u, delta_g2_after, delta_g2_before, cs.g2u);
  return run_checks(c, ops, checks, err, errcap);
}

// ---------------------------------------------------------------------------------------------
// process group (one GPU per process, e.g. under torchrun): the communicator of the cooperative calls
// ---------------------------------------------------------------------------------------------
int32_t sso_dist_unique_id(uint8_t out[128], char* err, size_t errcap) {
  const NcclApi* api = nccl_api(err, errcap);
  if (!api) return SSO_E_CUDA;
  ncclUniqueId id;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  NCCL_TRY(api, api->GetUniqueId(&id));
  memcpy(out, &id, 128);
  return SSO_OK;
}

int32_t sso_dist_init(int32_t rank, int32_t world, const uint8_t id128[128], int device, char* err, size_t errcap) {
  if (world < 1 || rank < 0 || rank >= world || !id128) { set_err(err, errcap, "bad process-group arguments"); return SSO_E_ARG; }
  const NcclApi* api = nccl_api(err, errcap);
  if (!api) return SSO_E_CUDA;
  std::lock_guard<std::mutex> g(dist_mutex());
  DistState& d = dist_state();
  if (d.on) { set_err(err, errcap, "process group already initialised"); return SSO_E_ARG; }
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess || device < 0 || device >= cnt) { set_err(err, errcap, "device %d out of range", device); return SSO_E_ARG; }
  int prev = 0;
  cudaGetDevice(&prev);
  CUDA_TRY(cudaSetDevice(device));
  ncclUniqueId id;
  memcpy(&id, id128, 128);
  NCCL_TRY(api, api->CommInitRank(&d.comm, world, id, rank));
  cudaSetDevice(prev);
  d.rank = rank; d.world = world; d.device = device; d.on = true; d.collectives = 0;
  return SSO_OK;
}

int32_t sso_dist_barrier(char* err, size_t errcap) {
  int32_t t;
  return dist_sum(0, &t, err, errcap);
}

int32_t sso_dist_finalize(void) {
  std::lock_guard<std::mutex> g(dist_mutex());
  DistState& d = dist_state();
  if (d.on) {
    char e[64];
    const NcclApi* api = nccl_api(e, sizeof e);
    if (api && d.comm) api->CommDestroy(d.comm);
    d = DistState();
  }
  return SSO_OK;
}

// out: [0] initialised, [1] rank, [2] world size, [3] all-gathers issued by the cooperative calls so far, [4] NCCL version
int32_t sso_dist_stats(uint64_t out[5]) {
  DistState& d = dist_state();
  out[0] = d.on; out[1] = (uint64_t)d.rank; out[2] = (uint64_t)d.world; out[3] = d.collectives; out[4] = 0;
  char e[64];
  const NcclApi* api = d.on || d.collectives ? nccl_api(e, sizeof e) : nullptr;
  int v = 0;
  if (api && api->GetVersion(&v) == ncclSuccess) out[4] = (uint64_t)v;
  return SSO_OK;
}

// every rank of a cooperative call must leave it with the same verdict: the failure flags are summed
static int32_t coop_result(bool coop, int32_t rc, char* err, size_t errcap) {
  if (!coop) return rc;
  int32_t total = 0;
  char e2[256];
  int32_t rc2 = dist_sum(rc != SSO_OK ? 1 : 0, &total, e2, sizeof e2);
  if (rc != SSO_OK) return rc;
  if (rc2 != SSO_OK) { set_err(err, errcap, "%s", e2); return rc2; }
  if (total != 0) { set_err(err, errcap, "another rank of the process group failed this call"); return SSO_E_VERIFY; }
  return SSO_OK;
}

// ---------------------------------------------------------------------------------------------
// generators
// ---------------------------------------------------------------------------------------------
int32_t sso_p1_set_generators(uint32_t curve, const uint8_t* g1_uncompressed, size_t g1_len, const uint8_t* g2_uncompressed, size_t g2_len,
                              int device, char* err, size_t errcap) {
  const CurveOps* ops = ops_for(curve);
  CurveSizes cs;
  if (!ops || !curve_sizes(curve, cs)) { set_err(err, errcap, "unknown curve %u", curve); return SSO_E_ARG; }
  if (!g1_uncompressed && !g2_uncompressed) {                       // back to the built-in constants
    std::lock_guard<std::mutex> g(gen_mutex());
    gen_override(curve) = GenOverride();
    return SSO_OK;
  }
  if (!g1_uncompressed || !g2_uncompressed || g1_len != cs.g1u || g2_len != cs.g2u) { set_err(err, errcap, "generators must be one uncompressed G1 point (%llu bytes) and one uncompressed G2 point (%llu bytes)", (unsigned long long)cs.g1u, (unsigned long long)cs.g2u); return SSO_E_ARG; }
  // a generator must be a non-zero point of the order-r subgroup
  Ctx c(err, errcap);
  int rc = c.init(device);
  if (rc) return rc;
  uint8_t* d_pts;
  uint32_t* d_status;
  if ((rc = c.alloc((void**)&d_pts, cs.g1u + cs.g2u))) return rc;
  if ((rc = status_buffer(c, &d_status, 0, true, err, errcap))) return rc;
  CUDA_TRY(cudaMemcpyAsync(d_pts, g1_uncompressed, cs.g1u, cudaMemcpyHostToDevice, c.s[0]));
  CUDA_TRY(cudaMemcpyAsync(d_pts + cs.g1u, g2_uncompressed, cs.g2u, cudaMemcpyHostToDevice, c.s[0]));
  if ((rc = ops->reencode(c, 0, GROUP_G1, d_pts, 0, 1, nullptr, 0, CHECK_FULL, 1, nullptr, d_status, err, errcap))) return rc;
  if ((rc = ops->reencode(c, 0, GROUP_G2, d_pts + cs.g1u, 0, 1, nullptr, 0, CHECK_FULL, 1, nullptr, d_status, err, errcap))) return rc;
  if ((rc = sync_all(c, err, errcap))) return rc;
  if ((rc = check_status(c, d_status, "generator", err, errcap))) return SSO_E_ARG;
  std::lock_guard<std::mutex> g(gen_mutex());
  GenOverride& o = gen_override(curve);
  o.g1u.assign(g1_uncompressed, g1_uncompressed + cs.g1u);
  o.g2u.assign(g2_uncompressed, g2_uncompressed + cs.g2u);
  o.set = true;
  return SSO_OK;
}

}  // extern "C" (kernel below)

// n copies of one serialized point
__global__ void k_fill_pattern(uint64_t n, const uint8_t* pattern, uint32_t size, uint8_t* out) {
  uint64_t total = n * size;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) out[i] = pattern[i % size];
}

namespace {
// n copies of the group generator into device memory (built-in constant or the caller's override)
int fill_generators(Ctx& c, int si, const CurveOps* ops, const CurveSizes& cs, uint32_t curve, uint32_t group, uint64_t n, uint8_t* d_out,
                    uint32_t out_compressed, char* err, size_t errcap) {
  if (n == 0) return SSO_OK;
  std::vector<uint8_t> pt;
  {
    std::lock_guard<std::mutex> g(gen_mutex());
    const GenOverride& o = gen_override(curve);
    if (o.set) pt = group == GROUP_G1 ? o.g1u : o.g2u;
  }
  if (pt.empty()) return ops->fill_generator(c, si, group, n, d_out, out_compressed, err, errcap);
  int rc;
  const size_t usz = point_size(cs, group, 0), osz = point_size(cs, group, out_compressed);
  uint8_t *d_u, *d_pat;
  uint32_t* d_status;
  if ((rc = c.alloc((void**)&d_u, usz, si))) return rc;
  if ((rc = c.alloc((void**)&d_pat, osz, si))) return rc;
  if ((rc = status_buffer(c, &d_status, si, false, err, errcap))) return rc;
  c.staging.emplace_back((usz + 3) / 4, 0u);
  memcpy(c.staging.back().data(), pt.data(), usz);
  CUDA_TRY(cudaMemcpyAsync(d_u, c.staging.back().data(), usz, cudaMemcpyHostToDevice, c.s[si]));
  if ((rc = ops->reencode(c, si, group, d_u, 0, 1, d_pat, out_compressed, CHECK_NO, 0, nullptr, d_status, err, errcap))) return rc;
  uint64_t total = n * osz;
  uint32_t blocks = (uint32_t)((total + 255) / 256 > 148 * 16 ? 148 * 16 : (total + 255) / 256);
  c.begin(PK_FILL, si, n);
  k_fill_pattern<<<blocks, 256, 0, c.s[si]>>>(n, d_pat, (uint32_t)osz, d_out);
  c.end(si);
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

bool is_coop(const sso_p1_params_t* p) { return p && p->contribution_mode == SSO_MODE_FULL && dist_state().on; }

// A file call with one mapped output of `out_size` bytes, made by every rank of the process group when `coop` (each computes
// its pieces into the shared mapping), else by this process alone.  The ranks agree after every step, so that a rank that
// failed makes the others return instead of waiting in a collective:
//   1. inputs() — every rank; then the lead rank creates the partial output
//   2. the other ranks map that partial output; then work(out) — every rank
//   3. the lead rank writes its small outputs with finish(outputs, out); every rank commits (the others only detach)
template <class Inputs, class Work, class Finish>
int32_t file_call(bool coop, const char* out_fn, size_t out_size, Inputs inputs, Work work, Finish finish, char* err, size_t errcap) {
  const bool lead = !coop || dist_state().rank == 0;
  Outputs outs;
  uint8_t* out = nullptr;
  int32_t rc = inputs();
  if (!rc && lead) rc = outs.create_mapped(out_fn, out_size, true, &out, err, errcap);
  if ((rc = coop_result(coop, rc, err, errcap))) return rc;
  if (!lead) rc = outs.create_mapped(out_fn, out_size, false, &out, err, errcap);
  if (!rc) rc = work(out);
  if ((rc = coop_result(coop, rc, err, errcap))) return rc;
  if (lead) rc = finish(outs, out);
  if (!rc) rc = outs.commit(err, errcap);
  return coop_result(coop, rc, err, errcap);
}
}  // namespace

extern "C" {

// phase1_cli::new_challenge(challenge_fn, challenge_hash_fn, params) — reference src/bin/new_setup.rs:105-109,
// src/bin/verify_transcript.rs:322-326: every element the generator, hash slot = Blake2b-512 of the empty string; writes the
// accumulator (uncompressed) and the 64 raw bytes of its hash
int32_t sso_p1_new_challenge_file(const char* challenge_fn, const char* challenge_hash_fn, const sso_p1_params_t* p, int device, char* err,
                                  size_t errcap) {
  P1Layout L;
  int rc = p1_layout(p, L, err, errcap);
  if (rc) return rc;
  if (!challenge_fn || !challenge_hash_fn) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  const CurveOps* ops = ops_for(p->curve);
  Outputs outs;
  uint8_t* out;
  if ((rc = outs.create_mapped(challenge_fn, L.acc_size, true, &out, err, errcap))) return rc;
  blake2b_512(nullptr, 0, out);
  const uint64_t counts[5] = {L.g1n, L.on, L.on, L.on, 1};
  static const uint32_t groups[5] = {GROUP_G1, GROUP_G2, GROUP_G1, GROUP_G1, GROUP_G2};
  {
    Ctx c(err, errcap);
    if ((rc = c.init(device < 0 ? 0 : device, 1))) return rc;
    const uint64_t piece = 1ull << 20;
    for (int v = 0; v < 5; v++) {
      const size_t usz = point_size(L.cs, groups[v], 0);
      for (uint64_t lo = 0; lo < counts[v]; lo += piece) {
        uint64_t cnt = lo + piece < counts[v] ? piece : counts[v] - lo;
        uint8_t* d_buf;
        if ((rc = c.alloc((void**)&d_buf, cnt * usz))) return rc;
        if ((rc = fill_generators(c, 0, ops, L.cs, p->curve, groups[v], cnt, d_buf, 0, err, errcap))) return rc;
        CUDA_TRY(cudaMemcpyAsync(out + L.off_u[v] + lo * usz, d_buf, cnt * usz, cudaMemcpyDeviceToHost, c.s[0]));
        if ((rc = c.recycle())) return rc;
      }
    }
  }
  if ((rc = outs.write_hash(challenge_hash_fn, out, L.acc_size, err, errcap))) return rc;
  return outs.commit(err, errcap);
}

// phase1_cli::contribute(challenge_fn, challenge_hash_fn, response_fn, response_hash_fn, check_input, batch_exp_mode, params, rng)
// — reference src/bin/contribute.rs:811-823, src/bin/verify_transcript.rs:678-696 (beacon, Full mode), src/bin/control.rs:793-808.
// rng -> the 32-byte seed of derive_rng_from_seed.  Full-mode calls with a process group are cooperative (every rank calls).
int32_t sso_p1_contribute_file(const sso_p1_params_t* p, const char* challenge_fn, const char* challenge_hash_fn,
                               const char* response_fn, const char* response_hash_fn, uint32_t check_input, uint32_t batch_exp_mode,
                               const uint8_t seed32[32], int device, char* err, size_t errcap) {
  (void)batch_exp_mode;                                    // outputs are mode-independent
  P1Layout L;
  int rc = p1_layout(p, L, err, errcap);
  if (rc) return rc;
  if (!challenge_fn || !challenge_hash_fn || !response_fn || !response_hash_fn || !seed32) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  if (!needs_streaming(p, L)) {
    // chunk-sized call: page-locked staging in and out (files.cuh), outputs written whole and renamed
    PinnedLease in(L.acc_size), out(L.contrib_size);
    if (!in.b.p || !out.b.p) { set_err(err, errcap, "cannot allocate page-locked staging buffers"); return SSO_E_CUDA; }
    if ((rc = refuse_existing(response_fn, err, errcap))) return rc;
    if ((rc = read_file_into(challenge_fn, in.b.p, L.acc_size, err, errcap))) return rc;
    if ((rc = contribute_buf_core(p, in.b.p, L.acc_size, out.b.p, L.contrib_size, nullptr, nullptr, nullptr, nullptr, 0, seed32, check_input, device, err, errcap))) return rc;
    Outputs outs;
    if ((rc = outs.write_whole(response_fn, out.b.p, L.contrib_size, err, errcap))) return rc;
    if ((rc = outs.write_whole(challenge_hash_fn, out.b.p, 64, err, errcap))) return rc;     // response[0..64) = hash(challenge)
    if ((rc = outs.write_hash(response_hash_fn, out.b.p, L.contrib_size, err, errcap))) return rc;
    return outs.commit(err, errcap);
  }
  MappedFile in;
  return file_call(is_coop(p), response_fn, L.contrib_size,
      [&]() -> int32_t {
        int32_t rc;
        if ((rc = in.open_ro(challenge_fn, err, errcap))) return rc;
        if (in.len != L.acc_size) { set_err(err, errcap, "The size of challenge file should be correct: %zu != %llu", in.len, (unsigned long long)L.acc_size); return SSO_E_ARG; }
        return SSO_OK;
      },
      [&](uint8_t* out) {
        return contribute_buf_core(p, in.p, in.len, out, L.contrib_size, nullptr, nullptr, nullptr, nullptr, 0, seed32, check_input, device, err, errcap);
      },
      [&](Outputs& outs, const uint8_t* out) {
        int32_t rc;
        if ((rc = outs.write_whole(challenge_hash_fn, out, 64, err, errcap))) return rc;        // response[0..64) = hash(challenge)
        return outs.write_hash(response_hash_fn, out, L.contrib_size, err, errcap);
      }, err, errcap);
}

// phase1_cli::transform_pok_and_correctness(challenge_fn, challenge_hash_fn, check_input, response_fn, response_hash_fn,
//                                           check_output, new_challenge_fn, new_challenge_hash_fn, subgroup_check_mode, ratio_check, params)
// — reference src/bin/contribute.rs:968-986, src/bin/verify_transcript.rs:466-484, 746-776 (Full mode), src/bin/control.rs:841-865
int32_t sso_p1_verify_chunk_file(const sso_p1_params_t* p, const char* challenge_fn, const char* challenge_hash_fn, uint32_t check_input,
                                 const char* response_fn, const char* response_hash_fn, uint32_t check_output,
                                 const char* new_challenge_fn, const char* new_challenge_hash_fn, uint32_t subgroup_check_mode,
                                 uint32_t ratio_check, int device, char* err, size_t errcap) {
  P1Layout L;
  int rc = p1_layout(p, L, err, errcap);
  if (rc) return rc;
  if (!challenge_fn || !challenge_hash_fn || !response_fn || !response_hash_fn || !new_challenge_fn || !new_challenge_hash_fn) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  if (!needs_streaming(p, L)) {
    PinnedLease chb(L.acc_size), respb(L.contrib_size), outb(L.acc_size);
    if (!chb.b.p || !respb.b.p || !outb.b.p) { set_err(err, errcap, "cannot allocate page-locked staging buffers"); return SSO_E_CUDA; }
    if ((rc = refuse_existing(new_challenge_fn, err, errcap))) return rc;
    if ((rc = read_file_into(challenge_fn, chb.b.p, L.acc_size, err, errcap))) return rc;
    if ((rc = read_file_into(response_fn, respb.b.p, L.contrib_size, err, errcap))) return rc;
    uint8_t ch_hash[64];
    if ((rc = verify_chunk_core(p, chb.b.p, L.acc_size, respb.b.p, L.contrib_size, outb.b.p, L.acc_size, check_input, check_output, subgroup_check_mode,
                                ratio_check, nullptr, device, ch_hash, err, errcap))) return rc;
    Outputs outs;
    if ((rc = outs.write_whole(new_challenge_fn, outb.b.p, L.acc_size, err, errcap))) return rc;
    if ((rc = outs.write_whole(challenge_hash_fn, ch_hash, 64, err, errcap))) return rc;
    if ((rc = outs.write_whole(response_hash_fn, outb.b.p, 64, err, errcap))) return rc;        // new_challenge[0..64) = hash(response)
    if ((rc = outs.write_hash(new_challenge_hash_fn, outb.b.p, L.acc_size, err, errcap))) return rc;
    return outs.commit(err, errcap);
  }
  MappedFile ch, resp;
  uint8_t ch_hash[64];
  return file_call(is_coop(p), new_challenge_fn, L.acc_size,
      [&]() -> int32_t {
        int32_t rc;
        if ((rc = ch.open_ro(challenge_fn, err, errcap))) return rc;
        if ((rc = resp.open_ro(response_fn, err, errcap))) return rc;
        if (ch.len != L.acc_size) { set_err(err, errcap, "The size of challenge file should be correct: %zu != %llu", ch.len, (unsigned long long)L.acc_size); return SSO_E_ARG; }
        if (resp.len != L.contrib_size) { set_err(err, errcap, "The size of response file should be correct: %zu != %llu", resp.len, (unsigned long long)L.contrib_size); return SSO_E_ARG; }
        return SSO_OK;
      },
      [&](uint8_t* out) {
        return verify_chunk_core(p, ch.p, ch.len, resp.p, resp.len, out, L.acc_size, check_input, check_output, subgroup_check_mode, ratio_check,
                                 nullptr, device, ch_hash, err, errcap);
      },
      [&](Outputs& outs, const uint8_t* out) {
        int32_t rc;
        if ((rc = outs.write_whole(challenge_hash_fn, ch_hash, 64, err, errcap))) return rc;
        if ((rc = outs.write_whole(response_hash_fn, out, 64, err, errcap))) return rc;         // new_challenge[0..64) = hash(response)
        return outs.write_hash(new_challenge_hash_fn, out, L.acc_size, err, errcap);
      }, err, errcap);
}

// phase1_cli::combine(response_list_fn, combined_fn, params) — reference src/bin/verify_transcript.rs:603-607,
// src/bin/control.rs:564-568.  `params` are the chunk-0 parameters of the ceremony (as the reference passes them); the list file
// names one response (compressed + public key) per chunk, in chunk order.  Output: the Full-mode accumulator, uncompressed, hash
// slot zero ([UP] Phase1::aggregation writes the vectors only).  devices / ndev: the GPUs of this process to decode on (NULL / 0 =
// `device`); with a process group every rank decodes its share of the pieces into the shared mapping.
int32_t sso_p1_combine_file(const char* response_list_fn, const char* combined_fn, const sso_p1_params_t* p, const int* devices, int ndev,
                            int device, char* err, size_t errcap) {
  if (!response_list_fn || !combined_fn || !p) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  sso_p1_params_t full = *p;
  full.contribution_mode = SSO_MODE_FULL; full.chunk_index = 0;
  P1Layout LF;
  int rc = p1_layout(&full, LF, err, errcap);
  if (rc) return rc;
  if (p->chunk_size == 0) { set_err(err, errcap, "combine needs the chunk size of the ceremony"); return SSO_E_ARG; }
  const CurveOps* ops = ops_for(p->curve);
  // the list of response files
  std::vector<std::string> names;
  {
    MappedFile txt;
    if ((rc = txt.open_ro(response_list_fn, err, errcap))) return rc;
    std::string cur;
    for (size_t i = 0; i < txt.len; i++) {
      const char ch = (char)txt.p[i];
      if (ch == '\n' || ch == '\r') { if (!cur.empty()) names.push_back(cur); cur.clear(); }
      else cur.push_back(ch);
    }
    if (!cur.empty()) names.push_back(cur);
  }
  const uint64_t nchunks = (LF.powers_g1_length + p->chunk_size - 1) / p->chunk_size;
  if (names.size() != nchunks) { set_err(err, errcap, "response list names %zu files, the ceremony has %llu chunks", names.size(), (unsigned long long)nchunks); return SSO_E_ARG; }
  std::vector<std::unique_ptr<MappedFile>> ins(nchunks);
  static const uint32_t groups[5] = {GROUP_G1, GROUP_G2, GROUP_G1, GROUP_G1, GROUP_G2};
  static const char* vnames[5] = {"tau_g1", "tau_g2", "alpha_g1", "beta_g1", "beta_g2"};
  return file_call(dist_state().on, combined_fn, LF.acc_size, [] { return (int32_t)SSO_OK; },
      [&](uint8_t* out) -> int32_t {
        int32_t rc;
        std::vector<RVec> vecs;
        for (uint64_t k = 0; k < nchunks; k++) {
          sso_p1_params_t pk = *p;
          pk.contribution_mode = SSO_MODE_CHUNKED; pk.chunk_index = k;
          P1Layout L;
          if ((rc = p1_layout(&pk, L, err, errcap))) return rc;
          ins[k].reset(new MappedFile());
          if ((rc = ins[k]->open_ro(names[k].c_str(), err, errcap))) return rc;
          if (ins[k]->len != L.contrib_size) { set_err(err, errcap, "The size of response file %s should be correct: %zu != %llu", names[k].c_str(), ins[k]->len, (unsigned long long)L.contrib_size); return SSO_E_ARG; }
          const uint64_t counts[5] = {L.g1n, L.on, L.on, L.on, k == 0 ? 1ull : 0ull};       // beta_g2 is taken from the first chunk
          for (int v = 0; v < 5; v++) {
            if (counts[v] == 0) continue;
            const size_t usz = point_size(L.cs, groups[v], 0);
            vecs.push_back({groups[v], ins[k]->p + L.off_c[v], 1, counts[v], out + LF.off_u[v] + (v == 4 ? 0 : L.start * usz), 0, 0,
                            CHECK_NO, 0, 0, vnames[v]});
          }
        }
        Participants P;
        if ((rc = resolve_participants(devices, ndev, device, true, P, err, errcap))) return rc;
        return stream_reencode(ops, LF.cs, vecs, p->batch_size, nullptr, 0, P, nullptr, err, errcap);
      },
      [](Outputs&, uint8_t* out) { memset(out, 0, 64); return (int32_t)SSO_OK; }, err, errcap);
}

// phase1_cli::transform_ratios(response_fn, check_input, params) — reference src/bin/verify_transcript.rs:646-653, 811-822,
// src/bin/control.rs:587-591, 866-873: consistency of a whole (Full-mode, uncompressed) accumulator.  Element 0 of tau_g1 /
// tau_g2 must be the generators; power_pairs(tau_g1), power_pairs(alpha_g1), power_pairs(beta_g1) against (tau_g2[0], tau_g2[1]);
// power_pairs(tau_g2) against (tau_g1[0], tau_g1[1]); beta_g2 against beta_g1[0].  The vectors are streamed in pieces over the
// participants (devices / ndev of this process, or the ranks of the process group); the per-participant partial sums are
// exchanged with ONE all-gather and added.  rlc_seed32: NULL (fresh entropy) outside tests.
int32_t sso_p1_verify_ratios_file(const sso_p1_params_t* p, const char* combined_fn, uint32_t check_input, const int* devices, int ndev,
                                  int device, const uint8_t* rlc_seed32, char* err, size_t errcap) {
  if (!p || !combined_fn) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  sso_p1_params_t full = *p;
  full.contribution_mode = SSO_MODE_FULL; full.chunk_index = 0;
  P1Layout L;
  int rc = p1_layout(&full, L, err, errcap);
  if (rc) return rc;
  const CurveOps* ops = ops_for(p->curve);
  const bool coop = dist_state().on;
  const size_t g1u = L.cs.g1u, g2u = L.cs.g2u;
  auto body = [&]() -> int32_t {
    int32_t rc;
    MappedFile in;
    if ((rc = in.open_ro(combined_fn, err, errcap))) return rc;
    if (in.len != L.acc_size) { set_err(err, errcap, "The size of the combined file should be correct: %zu != %llu", in.len, (unsigned long long)L.acc_size); return SSO_E_ARG; }
    Participants P;
    if ((rc = resolve_participants(devices, ndev, device, true, P, err, errcap))) return rc;
    const uint64_t counts[5] = {L.g1n, L.on, L.on, L.on, 1};
    static const uint32_t groups[5] = {GROUP_G1, GROUP_G2, GROUP_G1, GROUP_G1, GROUP_G2};
    static const char* vnames[5] = {"tau_g1", "tau_g2", "alpha_g1", "beta_g1", "beta_g2"};
    // transform_ratios deserialises with the caller's CheckForCorrectness; the pairings below need curve points, so the
    // on-curve test runs whatever the setting (uncompressed input)
    const uint32_t check = check_input == CHECK_NO ? (uint32_t)CHECK_NONZERO : check_input;
    std::vector<RVec> vecs;
    for (int v = 0; v < 5; v++)
      vecs.push_back({groups[v], in.p + L.off_u[v], 0, counts[v], nullptr, 0, v < 4 ? 1u : 0u, CHECK_FULL, check == CHECK_FULL ? 1u : 0u,
                      TWEAK_P1_RATIOS | (uint64_t)v, vnames[v]});
    std::vector<std::vector<uint8_t>> pairs;
    if ((rc = stream_reencode(ops, L.cs, vecs, p->batch_size, rlc_seed32, 0, P, &pairs, err, errcap))) return rc == SSO_E_INPUT ? SSO_E_VERIFY : rc;
    Ctx c(err, errcap);
    if ((rc = c.init(P.devices[0], 1))) return rc;
    std::vector<uint8_t> gen(g1u + g2u);
    if ((rc = generator_bytes(c, ops, L.cs, p->curve, gen.data(), err, errcap))) return rc;
    const uint8_t *g1_0 = in.p + L.off_u[0], *g1_1 = g1_0 + g1u, *g2_0 = in.p + L.off_u[1], *g2_1 = g2_0 + g2u;
    if (memcmp(g1_0, gen.data(), g1u) != 0) { set_err(err, errcap, "tau_g1[0] is not the G1 generator"); return SSO_E_VERIFY; }
    if (memcmp(g2_0, gen.data() + g1u, g2u) != 0) { set_err(err, errcap, "tau_g2[0] is not the G2 generator"); return SSO_E_VERIFY; }
    std::vector<RatioCheck> checks;
    add_check(checks, "power ratio: tau_g1", pairs[0].data(), pairs[0].data() + g1u, g1u, g2_0, g2_1, g2u);
    add_check(checks, "power ratio: tau_g2", g1_0, g1_1, g1u, pairs[1].data(), pairs[1].data() + g2u, g2u);
    add_check(checks, "power ratio: alpha_g1", pairs[2].data(), pairs[2].data() + g1u, g1u, g2_0, g2_1, g2u);
    add_check(checks, "power ratio: beta_g1", pairs[3].data(), pairs[3].data() + g1u, g1u, g2_0, g2_1, g2u);
    add_check(checks, "beta_g1[0] vs beta_g2", g1_0, in.p + L.off_u[3], g1u, g2_0, in.p + L.off_u[4], g2u);
    return run_checks(c, ops, checks, err, errcap);
  };
  return coop_result(coop, body(), err, errcap);
}

// ---------------------------------------------------------------------------------------------
// phase 2 on the parameter container (p2.cuh)
// ---------------------------------------------------------------------------------------------
namespace {

// a^-1 mod p on canonical little-endian limbs (binary extended Euclid; p odd, 0 < a < p) — one inversion per contribution
bool host_mod_inverse(const uint32_t* a, const uint32_t* p, int L, uint32_t* out) {
  auto is_zero = [&](const std::vector<uint32_t>& x) { for (uint32_t w : x) if (w) return false; return true; };
  auto is_one = [&](const std::vector<uint32_t>& x) { if (x[0] != 1) return false; for (int i = 1; i < L; i++) if (x[i]) return false; return true; };
  auto ge = [&](const std::vector<uint32_t>& x, const std::vector<uint32_t>& y) { for (int i = L - 1; i >= 0; i--) { if (x[i] != y[i]) return x[i] > y[i]; } return true; };
  auto sub = [&](std::vector<uint32_t>& x, const std::vector<uint32_t>& y) { uint64_t b = 0; for (int i = 0; i < L; i++) { uint64_t d = (uint64_t)x[i] - y[i] - b; x[i] = (uint32_t)d; b = (d >> 32) & 1; } return b; };
  auto add = [&](std::vector<uint32_t>& x, const std::vector<uint32_t>& y) { uint64_t cy = 0; for (int i = 0; i < L; i++) { uint64_t d = (uint64_t)x[i] + y[i] + cy; x[i] = (uint32_t)d; cy = d >> 32; } return cy; };
  auto shr1 = [&](std::vector<uint32_t>& x, uint32_t top) { for (int i = 0; i < L - 1; i++) x[i] = (x[i] >> 1) | (x[i + 1] << 31); x[L - 1] = (x[L - 1] >> 1) | (top << 31); };
  std::vector<uint32_t> u(a, a + L), v(p, p + L), x1(L, 0), x2(L, 0), pm(p, p + L);
  if (is_zero(u)) return false;
  x1[0] = 1;
  auto halve = [&](std::vector<uint32_t>& x) { uint32_t cy = 0; if (x[0] & 1) cy = (uint32_t)add(x, pm); shr1(x, cy); };
  while (!is_one(u) && !is_one(v)) {
    while (!(u[0] & 1)) { shr1(u, 0); halve(x1); }
    while (!(v[0] & 1)) { shr1(v, 0); halve(x2); }
    if (ge(u, v)) { sub(u, v); if (sub(x1, x2)) add(x1, pm); }
    else { sub(v, u); if (sub(x2, x1)) add(x2, pm); }
  }
  const std::vector<uint32_t>& r = is_one(u) ? x1 : x2;
  memcpy(out, r.data(), (size_t)L * 4);
  return true;
}

// scalar * point for one serialized point (host in, host out)
int scalar_mul_one(Ctx& c, const CurveOps* ops, const CurveSizes& cs, uint32_t group, const uint8_t* pt, bool in_compressed, const uint8_t* scalar,
                   uint8_t* out_uncompressed, char* err, size_t errcap) {
  int rc;
  const size_t isz = point_size(cs, group, in_compressed), usz = point_size(cs, group, 0);
  uint8_t *d_in, *d_out;
  uint32_t *d_status, *d_table;
  if ((rc = c.alloc((void**)&d_in, isz))) return rc;
  if ((rc = c.alloc((void**)&d_out, usz))) return rc;
  if ((rc = status_buffer(c, &d_status, 0, false, err, errcap))) return rc;
  CUDA_TRY(cudaMemcpyAsync(d_in, pt, isz, cudaMemcpyHostToDevice, c.s[0]));
  std::vector<uint8_t> one(ops->fr_bytes, 0);
  one[0] = 1;
  const uint8_t* coeffs[TAU_COEFF_SLOTS] = {scalar, nullptr, nullptr};
  if ((rc = ops->tau_tables(c, 0, 0, one.data(), coeffs, &d_table, err, errcap))) return rc;
  VecBatch b = batch_of({seg(d_in, d_out, 1, 0, 1, 1)});
  if ((rc = ops->batch_exp(c, 0, group, b, in_compressed, d_table, 0, CHECK_NO, d_status, err, errcap))) return rc;
  CUDA_TRY(cudaMemcpyAsync(out_uncompressed, d_out, usz, cudaMemcpyDeviceToHost, c.s[0]));
  CUDA_TRY(cudaStreamSynchronize(c.s[0]));
  return check_status(c, d_status, "point", err, errcap);
}

// r = hash_to_g2(transcript[..32]) and optionally r_delta
int p2_hash_to_g2(Ctx& c, const CurveOps* ops, const CurveSizes& cs, const uint8_t transcript[64], const uint32_t* d_scalar, uint8_t* r_out,
                  uint8_t* r_delta_out, char* err, size_t errcap) {
  int rc;
  uint32_t* d_seed;
  uint8_t *d_r, *d_rd;
  if ((rc = c.alloc((void**)&d_seed, 32))) return rc;
  if ((rc = c.alloc((void**)&d_r, cs.g2u))) return rc;
  if ((rc = c.alloc((void**)&d_rd, cs.g2u))) return rc;
  c.staging.emplace_back(8, 0u);
  memcpy(c.staging.back().data(), transcript, 32);
  CUDA_TRY(cudaMemcpyAsync(d_seed, c.staging.back().data(), 32, cudaMemcpyHostToDevice, c.s[0]));
  if ((rc = ops->hash_to_g2(c, 0, 1, d_seed, d_scalar, d_r, d_scalar ? d_rd : nullptr, err, errcap))) return rc;
  CUDA_TRY(cudaMemcpyAsync(r_out, d_r, cs.g2u, cudaMemcpyDeviceToHost, c.s[0]));
  if (d_scalar) CUDA_TRY(cudaMemcpyAsync(r_delta_out, d_rd, cs.g2u, cudaMemcpyDeviceToHost, c.s[0]));
  CUDA_TRY(cudaStreamSynchronize(c.s[0]));
  return SSO_OK;
}

}  // namespace

// phase2_cli::contribute on host buffers: challenge (uncompressed container) -> response (compressed container, one more
// contribution).  *response_len receives the size; SSO_E_ARG with the needed size in *response_len when response_cap is too small.
int32_t sso_p2_contribute_buf(uint32_t curve, const uint8_t* challenge, size_t challenge_len, uint8_t* response, size_t response_cap,
                              size_t* response_len, const uint8_t seed32[32], uint32_t check_input, int device, char* err, size_t errcap) {
  const CurveOps* ops = ops_for(curve);
  CurveSizes cs;
  if (!ops || !curve_sizes(curve, cs) || !challenge || !response_len || !seed32) { set_err(err, errcap, "unknown curve %u or null argument", curve); return SSO_E_ARG; }
  P2View vi;
  int rc = p2_parse(challenge, challenge_len, false, cs, vi, err, errcap);
  if (rc) return rc;
  const size_t need = p2_size(vi, cs, true, 1);
  *response_len = need;
  if (!response || response_cap < need) { set_err(err, errcap, "response buffer too small: %zu bytes needed", need); return SSO_E_ARG; }
  Ctx c(err, errcap);
  if ((rc = c.init(device, 1))) return rc;
  // the key pair: delta <- Fr::rand, s <- G1::rand, s_delta (the RNG draws, in the reference's order)
  std::vector<uint8_t> delta(cs.fr);
  KeygenState keys;
  if ((rc = keygen_stage1(c, 0, ops, cs, seed32, 1, keys, delta.data(), err, errcap))) return rc;
  if ((rc = keygen_collect_g1(c, 0, cs, keys, err, errcap))) return rc;
  FftDomain fr;                                             // the scalar field's modulus
  fft_domain(curve, fr);
  std::vector<uint32_t> dw(fr.L, 0), iw(fr.L, 0);
  memcpy(dw.data(), delta.data(), cs.fr);
  if (!host_mod_inverse(dw.data(), fr.modulus, (int)fr.L, iw.data())) { set_err(err, errcap, "delta is zero"); return SSO_E_INPUT; }
  std::vector<uint8_t> delta_inv(cs.fr);
  memcpy(delta_inv.data(), iw.data(), cs.fr);
  uint8_t transcript[64];
  p2_transcript(challenge, vi, keys.g1.data(), cs.g1u, transcript);
  std::vector<uint8_t> r(cs.g2u), r_delta(cs.g2u), delta_after(cs.g1u);
  if ((rc = p2_hash_to_g2(c, ops, cs, transcript, keys.d_scalars, r.data(), r_delta.data(), err, errcap))) return rc;
  if ((rc = scalar_mul_one(c, ops, cs, GROUP_G1, challenge + vi.delta_g1, false, delta.data(), delta_after.data(), err, errcap))) return rc;
  // the elements: h / l queries by delta^-1, delta_g1 / delta_g2 by delta, everything else re-encoded
  if ((rc = p2_transform(c, ops, cs, challenge, vi, response, true, delta.data(), delta_inv.data(), check_input, 0, "challenge", err, errcap))) return rc;
  // append the public key
  uint8_t* tail = response + need - vi.contrib_size;
  wr_u32be(response + need - 4 - (size_t)(vi.n_contrib + 1) * vi.contrib_size, vi.n_contrib + 1);
  memcpy(tail, delta_after.data(), cs.g1u);
  memcpy(tail + cs.g1u, keys.g1.data(), 2 * cs.g1u);
  memcpy(tail + 3 * cs.g1u, r_delta.data(), cs.g2u);
  memcpy(tail + 3 * cs.g1u + cs.g2u, transcript, 64);
  return SSO_OK;
}

// phase2_cli::verify on host buffers: challenge (uncompressed) + response (compressed) -> new challenge (uncompressed).
int32_t sso_p2_verify_buf(uint32_t curve, const uint8_t* challenge, size_t challenge_len, const uint8_t* response, size_t response_len,
                          uint8_t* new_challenge, size_t new_challenge_cap, size_t* new_challenge_len, uint32_t check_input, uint32_t check_output,
                          uint32_t subgroup_check_mode, const uint8_t* rlc_seed32, int device, char* err, size_t errcap) {
  const CurveOps* ops = ops_for(curve);
  CurveSizes cs;
  if (!ops || !curve_sizes(curve, cs) || !challenge || !response || !new_challenge_len) { set_err(err, errcap, "unknown curve %u or null argument", curve); return SSO_E_ARG; }
  P2View vc, vr;
  int rc;
  if ((rc = p2_parse(challenge, challenge_len, false, cs, vc, err, errcap))) return rc;
  if ((rc = p2_parse(response, response_len, true, cs, vr, err, errcap))) return rc == SSO_E_INPUT ? SSO_E_VERIFY : rc;
  const size_t need = p2_size(vr, cs, false, 0);
  *new_challenge_len = need;
  if (!new_challenge || new_challenge_cap < need) { set_err(err, errcap, "new challenge buffer too small: %zu bytes needed", need); return SSO_E_ARG; }
  auto reject = [&](const char* why) { set_err(err, errcap, "phase-2 verification: %s", why); return (int32_t)SSO_E_VERIFY; };
  if (vc.gamma_abc.n != vr.gamma_abc.n || vc.a_query.n != vr.a_query.n || vc.b_g1_query.n != vr.b_g1_query.n || vc.b_g2_query.n != vr.b_g2_query.n ||
      vc.h_query.n != vr.h_query.n || vc.l_query.n != vr.l_query.n) return reject("the query lengths changed");
  if (vr.n_contrib != vc.n_contrib + 1) return reject("the response must hold exactly one more contribution");
  if (memcmp(challenge + vc.cs_hash, response + vr.cs_hash, 64) != 0) return reject("cs_hash changed");
  if (memcmp(challenge + vc.contribs, response + vr.contribs, (size_t)vc.n_contrib * vc.contrib_size) != 0) return reject("earlier contributions changed");
  Ctx c(err, errcap);
  if ((rc = c.init(device, 1))) return rc;
  // Groth16 queries may hold the point at infinity (unused variables): the zero test follows check_output here
  const uint32_t elem_check = check_output, subgroup = verify_subgroup(check_output, subgroup_check_mode);
  if (check_input != CHECK_NO) {
    std::vector<uint8_t> scratch(p2_size(vc, cs, false, 0));
    if ((rc = p2_transform(c, ops, cs, challenge, vc, scratch.data(), false, nullptr, nullptr, check_input, check_input == CHECK_FULL ? 1u : 0u, "challenge", err, errcap)))
      return rc == SSO_E_INPUT ? SSO_E_VERIFY : rc;
  }
  if ((rc = p2_transform(c, ops, cs, response, vr, new_challenge, false, nullptr, nullptr, elem_check, subgroup, "response", err, errcap)))
    return rc == SSO_E_INPUT ? SSO_E_VERIFY : rc;
  P2View vn;
  if ((rc = p2_parse(new_challenge, need, false, cs, vn, err, errcap))) return rc;
  // untouched elements
  std::vector<P2Item> ic = p2_items(vc), in_ = p2_items(vn);
  for (size_t i = 0; i < ic.size(); i++) {
    if (ic[i].kind != 0) continue;
    const size_t usz = point_size(cs, ic[i].group, 0);
    if (memcmp(challenge + ic[i].off, new_challenge + in_[i].off, ic[i].n * usz) != 0) return reject("an element outside h_query / l_query / delta changed");
  }
  // the public key of this contribution
  const uint8_t* pk = response + vr.contribs + (size_t)vc.n_contrib * vr.contrib_size;
  const uint8_t *delta_after = pk, *s_pair = pk + cs.g1u, *r_delta = pk + 3 * cs.g1u, *pk_transcript = pk + 3 * cs.g1u + cs.g2u;
  {
    uint8_t* d_pk;
    uint32_t* d_status;
    if ((rc = c.alloc((void**)&d_pk, vr.contrib_size))) return rc;
    if ((rc = status_buffer(c, &d_status, 0, true, err, errcap))) return rc;
    CUDA_TRY(cudaMemcpyAsync(d_pk, pk, vr.contrib_size, cudaMemcpyHostToDevice, c.s[0]));
    if ((rc = ops->reencode(c, 0, GROUP_G1, d_pk, 0, 3, nullptr, 0, CHECK_FULL, 1, nullptr, d_status, err, errcap))) return rc;
    if ((rc = ops->reencode(c, 0, GROUP_G2, d_pk + 3 * cs.g1u, 0, 1, nullptr, 0, CHECK_FULL, 1, nullptr, d_status, err, errcap))) return rc;
    CUDA_TRY(cudaStreamSynchronize(c.s[0]));
    if ((rc = check_status(c, d_status, "public key", err, errcap))) return rc == SSO_E_INPUT ? SSO_E_VERIFY : rc;
  }
  uint8_t transcript[64];
  p2_transcript(challenge, vc, s_pair, cs.g1u, transcript);
  if (memcmp(transcript, pk_transcript, 64) != 0) return reject("the transcript hash of the public key does not continue the challenge");
  if (memcmp(delta_after, new_challenge + vn.delta_g1, cs.g1u) != 0) return reject("delta_after of the public key is not the new delta_g1");
  std::vector<uint8_t> r(cs.g2u);
  if ((rc = p2_hash_to_g2(c, ops, cs, transcript, nullptr, r.data(), nullptr, err, errcap))) return rc;
  std::vector<RatioCheck> checks;
  add_check(checks, "proof of knowledge: delta", s_pair, s_pair + cs.g1u, cs.g1u, r.data(), r_delta, cs.g2u);
  add_check(checks, "delta_g1 vs delta proof", challenge + vc.delta_g1, new_challenge + vn.delta_g1, cs.g1u, r.data(), r_delta, cs.g2u);
  add_check(checks, "delta_g1 vs delta_g2", challenge + vc.delta_g1, new_challenge + vn.delta_g1, cs.g1u, challenge + vc.delta_g2, new_challenge + vn.delta_g2, cs.g2u);
  // the queries: merge_pairs(before, after) against (delta_g2 after, delta_g2 before)
  std::vector<uint8_t> pairs[2];
  const P2Vec* qb[2] = {&vc.h_query, &vc.l_query};
  const P2Vec* qa[2] = {&vn.h_query, &vn.l_query};
  static const char* qn[2] = {"h_query vs delta_g2", "l_query vs delta_g2"};
  for (int q = 0; q < 2; q++) {
    const uint64_t n = qb[q]->n;
    if (n == 0) continue;
    if (n > (1ull << 24)) return reject("query longer than 2^24 elements");
    uint8_t *d_b, *d_a;
    uint32_t* d_status;
    if ((rc = status_buffer(c, &d_status, 0, true, err, errcap))) return rc;
    if ((rc = c.alloc((void**)&d_b, n * cs.g1u))) return rc;
    if ((rc = c.alloc((void**)&d_a, n * cs.g1u))) return rc;
    CUDA_TRY(cudaMemcpyAsync(d_b, challenge + qb[q]->off, n * cs.g1u, cudaMemcpyHostToDevice, c.s[0]));
    CUDA_TRY(cudaMemcpyAsync(d_a, new_challenge + qa[q]->off, n * cs.g1u, cudaMemcpyHostToDevice, c.s[0]));
    const uint64_t tweak[4] = {TWEAK_P2_VERIFY | (uint64_t)q, n, 0, 0};
    pairs[q].resize(2 * cs.g1u);
    if ((rc = pair_to_host(c, ops, GROUP_G1, cs.g1u, n, {d_b, 0, CHECK_NO, 0}, {d_a, 0, CHECK_NO, 0}, rlc_seed32, tweak, d_status, "query",
                           pairs[q].data(), err, errcap))) return rc == SSO_E_INPUT ? SSO_E_VERIFY : rc;
    add_check(checks, qn[q], pairs[q].data(), pairs[q].data() + cs.g1u, cs.g1u, new_challenge + vn.delta_g2, challenge + vc.delta_g2, cs.g2u);
  }
  return run_checks(c, ops, checks, err, errcap);
}

// phase2_cli::contribute::<P>(challenge_fn, challenge_hash_fn, response_fn, response_hash_fn, check_input, batch_exp_mode, rng)
// — reference src/bin/contribute.rs:827-838; the curve type parameter becomes `curve`, the rng its 32-byte seed
int32_t sso_p2_contribute_file(uint32_t curve, const char* challenge_fn, const char* challenge_hash_fn, const char* response_fn,
                               const char* response_hash_fn, uint32_t check_input, uint32_t batch_exp_mode, const uint8_t seed32[32], int device,
                               char* err, size_t errcap) {
  (void)batch_exp_mode;
  if (!challenge_fn || !challenge_hash_fn || !response_fn || !response_hash_fn || !seed32) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  MappedFile in;
  Outputs outs;
  uint8_t* out;
  int rc;
  if ((rc = in.open_ro(challenge_fn, err, errcap))) return rc;
  size_t need = 0;
  rc = sso_p2_contribute_buf(curve, in.p, in.len, nullptr, 0, &need, seed32, check_input, device, err, errcap);
  if (rc != SSO_E_ARG || need == 0) return rc ? rc : SSO_E_ARG;
  if ((rc = outs.create_mapped(response_fn, need, true, &out, err, errcap))) return rc;
  if ((rc = sso_p2_contribute_buf(curve, in.p, in.len, out, need, &need, seed32, check_input, device, err, errcap))) return rc;
  if ((rc = outs.write_hash(challenge_hash_fn, in.p, in.len, err, errcap))) return rc;
  if ((rc = outs.write_hash(response_hash_fn, out, need, err, errcap))) return rc;
  return outs.commit(err, errcap);
}

// phase2_cli::verify::<P>(challenge_fn, challenge_hash_fn, check_input, response_fn, response_hash_fn, check_output, new_challenge_fn,
//                         new_challenge_hash_fn, subgroup_check_mode, verify_full) — reference src/bin/contribute.rs:990-1007
int32_t sso_p2_verify_file(uint32_t curve, const char* challenge_fn, const char* challenge_hash_fn, uint32_t check_input, const char* response_fn,
                           const char* response_hash_fn, uint32_t check_output, const char* new_challenge_fn, const char* new_challenge_hash_fn,
                           uint32_t subgroup_check_mode, uint32_t verify_full, int device, char* err, size_t errcap) {
  (void)verify_full;                                       // this container is always the full parameter set
  if (!challenge_fn || !challenge_hash_fn || !response_fn || !response_hash_fn || !new_challenge_fn || !new_challenge_hash_fn) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  MappedFile ch, resp;
  Outputs outs;
  uint8_t* out;
  int rc;
  if ((rc = ch.open_ro(challenge_fn, err, errcap))) return rc;
  if ((rc = resp.open_ro(response_fn, err, errcap))) return rc;
  size_t need = 0;
  rc = sso_p2_verify_buf(curve, ch.p, ch.len, resp.p, resp.len, nullptr, 0, &need, check_input, check_output, subgroup_check_mode, nullptr, device, err, errcap);
  if (rc != SSO_E_ARG || need == 0) return rc ? rc : SSO_E_ARG;
  if ((rc = outs.create_mapped(new_challenge_fn, need, true, &out, err, errcap))) return rc;
  if ((rc = sso_p2_verify_buf(curve, ch.p, ch.len, resp.p, resp.len, out, need, &need, check_input, check_output, subgroup_check_mode, nullptr, device, err, errcap))) return rc;
  if ((rc = outs.write_hash(challenge_hash_fn, ch.p, ch.len, err, errcap))) return rc;
  if ((rc = outs.write_hash(response_hash_fn, resp.p, resp.len, err, errcap))) return rc;
  if ((rc = outs.write_hash(new_challenge_hash_fn, out, need, err, errcap))) return rc;
  return outs.commit(err, errcap);
}

// ---------------------------------------------------------------------------------------------
// prepare_phase2 (p2prep.cuh)
// ---------------------------------------------------------------------------------------------
// Radix-2 group FFT over the scalar field's two-adic domain — the primitive of phase2_cli::prepare_phase2
// (ark-poly Radix2EvaluationDomain::ifft / fft applied to curve points, reference src/bin/intermediate_transform.rs:213-226).
int32_t sso_group_fft_dev(uint32_t curve, uint32_t group, const void* d_in, uint32_t in_compressed, uint32_t log_n, uint32_t inverse,
                          void* d_out, uint32_t out_compressed, int device, char* err, size_t errcap) {
  const CurveOps* ops = ops_for(curve);
  FftDomain d;
  if (!ops || !fft_domain(curve, d)) { set_err(err, errcap, "unknown curve %u", curve); return SSO_E_ARG; }
  Ctx c(err, errcap);
  int rc = c.init(device);
  if (rc) return rc;
  if (group > 1 || !d_in || !d_out) { set_err(err, errcap, "unknown group %u or null buffer", group); return SSO_E_ARG; }
  uint32_t* d_status;
  if ((rc = status_buffer(c, &d_status, 0, true, err, errcap))) return rc;
  CurveSizes cs;
  curve_sizes(curve, cs);
  const uint8_t* src = (const uint8_t*)d_in;
  if (in_compressed && log_n <= 24) {
    uint8_t* d_u;
    const uint64_t n = 1ull << log_n;
    if ((rc = c.alloc((void**)&d_u, n * point_size(cs, group, 0)))) return rc;
    if ((rc = ops->reencode(c, 0, group, src, 1, n, d_u, 0, CHECK_NO, 0, nullptr, d_status, err, errcap))) return rc;
    src = d_u;
  }
  std::vector<uint8_t> minv;
  if (inverse) minv = fft_inv_size(d, log_n, ops->fr_bytes);
  if ((rc = ops->group_fft(c, 0, group, src, log_n, inverse ? d.root_inv : d.root, d.two_adicity, inverse ? minv.data() : nullptr,
                           (uint8_t*)d_out, out_compressed, d_status, err, errcap))) return rc;
  if ((rc = sync_all(c, err, errcap))) return rc;
  return check_status(c, d_status, "group FFT input", err, errcap);
}

// phase2_cli::prepare_phase2 on host buffers (reference src/bin/intermediate_transform.rs:213-226): a Full-mode accumulator
// (uncompressed) -> the Lagrange-basis Groth16Params of size phase2_size.  *out_len receives the size; SSO_E_ARG with the needed size
// in *out_len when out_cap is too small.
int32_t sso_p2_prepare_buf(const sso_p1_params_t* p, const uint8_t* accumulator, size_t len, uint64_t phase2_size, uint8_t* out, size_t out_cap,
                           size_t* out_len, int device, char* err, size_t errcap) {
  if (out_len) *out_len = 0;
  P1Layout L;
  FftDomain d;
  int log_m;
  int rc = p2prep_check(p, phase2_size, L, d, log_m, err, errcap);
  if (rc) return rc;
  if (!out_len) { set_err(err, errcap, "null out_len"); return SSO_E_ARG; }
  if (!accumulator || len != L.acc_size) { set_err(err, errcap, "accumulator is %zu bytes, the parameters give %llu", len, (unsigned long long)L.acc_size); return SSO_E_ARG; }
  const size_t need = p2prep_size(L.cs, phase2_size);
  *out_len = need;
  if (!out || out_cap < need) { set_err(err, errcap, "output buffer too small: %zu bytes needed", need); return SSO_E_ARG; }
  Ctx c(err, errcap);
  if ((rc = c.init(device, 2))) return rc;
  return p2_prepare(c, ops_for(p->curve), L, d, log_m, accumulator, out, err, errcap);
}

// phase2_cli::prepare_phase2(phase2_filename, response_filename, phase2_size, parameters) — reference
// src/bin/intermediate_transform.rs:213-226.  The output is created under a temporary name and renamed when the call succeeded.
int32_t sso_p2_prepare_file(const char* phase2_fn, const char* response_fn, uint64_t phase2_size, const sso_p1_params_t* p, int device,
                            char* err, size_t errcap) {
  if (!phase2_fn || !response_fn) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  P1Layout L;
  FftDomain d;
  int log_m;
  int rc = p2prep_check(p, phase2_size, L, d, log_m, err, errcap);
  if (rc) return rc;
  MappedFile in;
  Outputs outs;
  uint8_t* out;
  if ((rc = in.open_ro(response_fn, err, errcap))) return rc;
  size_t need = 0;
  rc = sso_p2_prepare_buf(p, in.p, in.len, phase2_size, nullptr, 0, &need, device, err, errcap);
  if (rc != SSO_E_ARG || need == 0) return rc ? rc : SSO_E_ARG;
  if ((rc = outs.create_mapped(phase2_fn, need, true, &out, err, errcap))) return rc;
  if ((rc = sso_p2_prepare_buf(p, in.p, in.len, phase2_size, out, need, &need, device, err, errcap))) return rc;
  return outs.commit(err, errcap);
}

// The group FFT in parts on host buffers (p2prep.cuh parts_fft): the transform of sso_group_fft_dev, uncompressed, for any number of
// parts and past 2^24 points, over the devices of this process.
int32_t sso_group_fft_parts_buf(uint32_t curve, uint32_t group, const uint8_t* in, size_t in_len, uint32_t log_n, uint32_t inverse,
                                uint8_t* out, size_t out_len, uint64_t parts, const int* devices, int ndev, int device, char* err, size_t errcap) {
  const CurveOps* ops = ops_for(curve);
  FftDomain d;
  CurveSizes cs;
  if (!ops || !fft_domain(curve, d) || !curve_sizes(curve, cs)) { set_err(err, errcap, "unknown curve %u", curve); return SSO_E_ARG; }
  if (group > 1) { set_err(err, errcap, "unknown group %u", group); return SSO_E_ARG; }
  if (log_n > d.two_adicity) { set_err(err, errcap, "group FFT of 2^%u points: beyond the radix-2 domain (2^%u)", log_n, d.two_adicity); return SSO_E_ARG; }
  const int log_p = log2_exact(parts);
  if (log_p < 0 || (uint32_t)log_p > log_n || log_n - (uint32_t)log_p > 24 || log_p > 24) {
    set_err(err, errcap, "%llu parts of 2^%u points: a power of two up to 2^24 and the number of points, with parts of at most 2^24 points",
            (unsigned long long)parts, log_n);
    return SSO_E_ARG;
  }
  const uint64_t n = 1ull << log_n;
  const size_t bytes = n * point_size(cs, group, 0);
  if (!in || !out || in_len != bytes || out_len != bytes) {
    set_err(err, errcap, "input and output must be %zu bytes each (2^%u uncompressed points)", bytes, log_n);
    return SSO_E_ARG;
  }
  if (in < out + out_len && out < in + in_len) { set_err(err, errcap, "the output must not overlap the input"); return SSO_E_ARG; }
  Participants Pt;
  int rc = resolve_participants(devices, ndev, device, false, Pt, err, errcap);
  if (rc) return rc;
  std::vector<uint8_t> minv;
  if (inverse) minv = fft_inv_size(d, log_n, ops->fr_bytes);
  const PartsPlan pl = parts_plan(log_n, (uint32_t)log_p, inverse ? d.root_inv : d.root, d.two_adicity, inverse ? minv.data() : nullptr);
  const PartsVec v = {group, in, out, 0};
  return parts_fft(ops, cs, pl, &v, 1, Pt, CHECK_NO, "group FFT input", 0, nullptr, err, errcap);
}

// prepare_phase2 in parts over the devices of this process (p2prep.cuh p2_prepare_devices): the output of sso_p2_prepare_buf, for
// every size the radix-2 domain and the accumulator allow.
int32_t sso_p2_prepare_devices_buf(const sso_p1_params_t* p, const uint8_t* accumulator, size_t len, uint64_t phase2_size, uint8_t* out,
                                   size_t out_cap, size_t* out_len, const int* devices, int ndev, int device, char* err, size_t errcap) {
  if (out_len) *out_len = 0;
  P1Layout L;
  FftDomain d;
  int log_m;
  int rc = p2prep_check(p, phase2_size, L, d, log_m, err, errcap, 64);
  if (rc) return rc;
  if (!out_len) { set_err(err, errcap, "null out_len"); return SSO_E_ARG; }
  if (!accumulator || len != L.acc_size) { set_err(err, errcap, "accumulator is %zu bytes, the parameters give %llu", len, (unsigned long long)L.acc_size); return SSO_E_ARG; }
  const size_t need = p2prep_size(L.cs, phase2_size);
  *out_len = need;
  if (!out || out_cap < need) { set_err(err, errcap, "output buffer too small: %zu bytes needed", need); return SSO_E_ARG; }
  return p2_prepare_devices(ops_for(p->curve), L, d, log_m, accumulator, out, devices, ndev, device, err, errcap);
}

// sso_p2_prepare_file in parts over the devices of this process.  The output (which holds the intermediate rows of the transform)
// is created under a temporary name and renamed when the call succeeded.
int32_t sso_p2_prepare_devices_file(const char* phase2_fn, const char* response_fn, uint64_t phase2_size, const sso_p1_params_t* p,
                                    const int* devices, int ndev, int device, char* err, size_t errcap) {
  if (!phase2_fn || !response_fn) { set_err(err, errcap, "null argument"); return SSO_E_ARG; }
  P1Layout L;
  FftDomain d;
  int log_m;
  int rc = p2prep_check(p, phase2_size, L, d, log_m, err, errcap, 64);
  if (rc) return rc;
  if ((rc = refuse_existing(phase2_fn, err, errcap))) return rc;
  MappedFile in;
  Outputs outs;
  uint8_t* out;
  if ((rc = in.open_ro(response_fn, err, errcap))) return rc;
  if (in.len != L.acc_size) { set_err(err, errcap, "accumulator is %zu bytes, the parameters give %llu", in.len, (unsigned long long)L.acc_size); return SSO_E_ARG; }
  if ((rc = outs.create_mapped(phase2_fn, p2prep_size(L.cs, phase2_size), true, &out, err, errcap))) return rc;
  if ((rc = p2_prepare_devices(ops_for(p->curve), L, d, log_m, in.p, out, devices, ndev, device, err, errcap))) return rc;
  return outs.commit(err, errcap);
}

int32_t sso_imad_peak(int device, int variant, double* macs_per_s, char* err, size_t errcap) {
  Ctx c(err, errcap);
  int rc = c.init(device);
  if (rc) return rc;
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  uint64_t* d_sink;
  if ((rc = c.alloc((void**)&d_sink, 8))) return rc;
  const uint32_t iters = 4096, threads = 256, blocks = prop.multiProcessorCount * 8;
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  double best = 0;
  for (int rep = 0; rep < 6; rep++) {
    CUDA_TRY(cudaEventRecord(e0, c.s[0]));
    k_imad_probe<<<blocks, threads, 0, c.s[0]>>>(iters, (uint32_t)variant, 12345u + rep, d_sink);
    CUDA_TRY(cudaEventRecord(e1, c.s[0]));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    double macs = (double)iters * 32.0 * threads * blocks;
    double rate = macs / (ms * 1e-3);
    if (rep > 0 && rate > best) best = rate;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *macs_per_s = best;
  return SSO_OK;
}

int32_t sso_test_field_mul(uint32_t field, const uint8_t* a, const uint8_t* b, uint8_t* out, uint64_t n, int device,
                           char* err, size_t errcap) {
  Ctx c(err, errcap);
  int rc = c.init(device);
  if (rc) return rc;
  static const size_t nbytes[5] = {32, 48, 96, 95, 95};
  if (field > 4) { set_err(err, errcap, "unknown field %u", field); return SSO_E_ARG; }
  size_t bytes = n * nbytes[field];
  uint8_t *d_a, *d_b, *d_o;
  uint32_t* d_status;
  if ((rc = c.alloc((void**)&d_a, bytes))) return rc;
  if ((rc = c.alloc((void**)&d_b, bytes))) return rc;
  if ((rc = c.alloc((void**)&d_o, bytes))) return rc;
  if ((rc = status_buffer(c, &d_status, 0, true, err, errcap))) return rc;
  CUDA_TRY(cudaMemcpyAsync(d_a, a, bytes, cudaMemcpyHostToDevice, c.s[0]));
  CUDA_TRY(cudaMemcpyAsync(d_b, b, bytes, cudaMemcpyHostToDevice, c.s[0]));
  uint32_t g = div_up(n, 128);
  switch (field) {
    case 0: k_test_field_mul<Fr253><<<g, 128, 0, c.s[0]>>>(d_a, d_b, d_o, (uint32_t)n, d_status); break;
    case 1: k_test_field_mul<Fq377><<<g, 128, 0, c.s[0]>>>(d_a, d_b, d_o, (uint32_t)n, d_status); break;
    case 2: k_test_field_mul<Fq761><<<g, 128, 0, c.s[0]>>>(d_a, d_b, d_o, (uint32_t)n, d_status); break;
    case 3: k_test_field_mul<Fq4><<<g, 128, 0, c.s[0]>>>(d_a, d_b, d_o, (uint32_t)n, d_status); break;
    case 4: k_test_field_mul<Fq6><<<g, 128, 0, c.s[0]>>>(d_a, d_b, d_o, (uint32_t)n, d_status); break;
  }
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(out, d_o, bytes, cudaMemcpyDeviceToHost, c.s[0]));
  if ((rc = sync_all(c, err, errcap))) return rc;
  return check_status(c, d_status, "field element", err, errcap);
}

int32_t sso_test_field_op(uint32_t field, const uint32_t* ops, const uint32_t* a, const uint32_t* b, const uint32_t* k, uint32_t* out,
                          uint32_t* rc, uint64_t n, int device, char* err, size_t errcap) {
  static const uint32_t words[11] = {8, 12, 24, 24, 24, 24, 48, 72, 24, 48, 72};     // per element, by field id
  if (field > 10) { set_err(err, errcap, "unknown field %u", field); return SSO_E_ARG; }
  Ctx c(err, errcap);
  int rc_ = c.init(device);
  if (rc_) return rc_;
  const size_t wbytes = n * words[field] * 4, nbytes = n * 4;
  uint32_t *d_ops, *d_a, *d_b, *d_k, *d_out, *d_rc;
  if ((rc_ = c.alloc((void**)&d_ops, nbytes))) return rc_;
  if ((rc_ = c.alloc((void**)&d_a, wbytes))) return rc_;
  if ((rc_ = c.alloc((void**)&d_b, wbytes))) return rc_;
  if ((rc_ = c.alloc((void**)&d_k, nbytes))) return rc_;
  if ((rc_ = c.alloc((void**)&d_out, wbytes))) return rc_;
  if ((rc_ = c.alloc((void**)&d_rc, nbytes))) return rc_;
  CUDA_TRY(cudaMemcpyAsync(d_ops, ops, nbytes, cudaMemcpyHostToDevice, c.s[0]));
  CUDA_TRY(cudaMemcpyAsync(d_a, a, wbytes, cudaMemcpyHostToDevice, c.s[0]));
  CUDA_TRY(cudaMemcpyAsync(d_b, b, wbytes, cudaMemcpyHostToDevice, c.s[0]));
  CUDA_TRY(cudaMemcpyAsync(d_k, k, nbytes, cudaMemcpyHostToDevice, c.s[0]));
  CUDA_TRY(cudaMemsetAsync(d_out, 0, wbytes, c.s[0]));
  CUDA_TRY(cudaMemsetAsync(d_rc, 0, nbytes, c.s[0]));
  if ((rc_ = run_field_op(c, 0, field, d_ops, d_a, d_b, d_k, d_out, d_rc, n, err, errcap))) return rc_;
  CUDA_TRY(cudaMemcpyAsync(out, d_out, wbytes, cudaMemcpyDeviceToHost, c.s[0]));
  CUDA_TRY(cudaMemcpyAsync(rc, d_rc, nbytes, cudaMemcpyDeviceToHost, c.s[0]));
  return sync_all(c, err, errcap);
}

}  // extern "C"
