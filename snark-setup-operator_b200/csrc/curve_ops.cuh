// Per-curve kernel instantiations behind a small function table, so that each curve compiles
// in its own translation unit (parallel nvcc) and abi.cu stays curve-agnostic.
#pragma once
#include <type_traits>
#include "host.cuh"
#include "kernels.cuh"
#include "msm.cuh"
#include "pairing.cuh"
#include "keygen.cuh"
#include "blake2b.h"
#include <cub/device/device_radix_sort.cuh>
#include <random>

namespace sso {

struct CurveOps {
  // K1: tau-power tables + coefficient slots for one call (shared by every vector of the call)
  int (*tau_tables)(Ctx& c, int si, uint64_t first_index, const uint8_t* tau, const uint8_t* const coeffs[TAU_COEFF_SLOTS],
                    uint32_t** d_table, char* err, size_t errcap);
  // K2-K4 on up to four vectors of one group in one launch pair
  int (*batch_exp)(Ctx& c, int si, uint32_t group, const VecBatch& batch, uint32_t in_compressed, const uint32_t* d_table,
                   uint32_t out_compressed, uint32_t check, uint32_t* d_status, char* err, size_t errcap);
  // K2-K4 for the G1 and G2 vectors of a chunk in one launch pair (tail filling across the groups)
  int (*batch_exp_chunk)(Ctx& c, int si, const VecBatch& b1, const VecBatch& b2, uint32_t in_compressed, const uint32_t* d_table,
                         uint32_t out_compressed, uint32_t check, uint32_t* d_status, char* err, size_t errcap);
  // K3 (+K6) alone
  int (*reencode)(Ctx& c, int si, uint32_t group, const uint8_t* d_in, uint32_t in_compressed, uint64_t n, uint8_t* d_out,
                  uint32_t out_compressed, uint32_t check, uint32_t subgroup, uint32_t* d_aff, uint32_t* d_status, char* err,
                  size_t errcap);
  // K5: (sum r_i a_i, sum r_i b_i) for two affine Montgomery point arrays ([point][x|y] words, zero = infinity) with
  // ChaCha20(seed32) scalars; writes the two points uncompressed to d_out (2 * uncompressed size bytes)
  // tweak (4 words, may be null): with a caller-supplied seed the ChaCha20 key of this MSM is Blake2b-256(seed32 || tweak),
  // so that the MSMs of one verification (vectors, chunks, pieces, ranks) never share their scalars; null = seed32 as is
  int (*msm_pairs)(Ctx& c, int si, uint32_t group, const uint32_t* d_aff_a, const uint32_t* d_aff_b, uint64_t n,
                   const uint8_t seed32[32], const uint64_t* tweak, uint8_t* d_out, char* err, size_t errcap);
  // K8: same_ratio verdicts for n checks laid out a | b | c | d (uncompressed); verdict 1 = equal ratios,
  // 0 = different, 0x100 + code = undecodable input
  int (*same_ratio)(Ctx& c, int si, const uint8_t* d_checks, uint64_t n, uint32_t* d_verdicts, char* err, size_t errcap);
  uint32_t check_bytes;
  // a3: key generation pieces.  keygen_g1: nscalars Fr::rand draws then, per scalar, g1_s <- G1::rand and
  // g1_s_x; d_scalars: nscalars * Fr words (canonical), d_g1: 2 * nscalars uncompressed G1 points.
  int (*keygen_g1)(Ctx& c, int si, const uint32_t* d_seed, uint32_t nscalars, uint32_t* d_scalars, uint8_t* d_g1, char* err, size_t errcap);
  // the private scalars alone (the first nscalars Fr::rand draws): microseconds, so that the main kernels of a contribution
  // can start while keygen_g1 (the single-thread point sampling and the proofs' G1 halves) runs beside them
  int (*keygen_scalars)(Ctx& c, int si, const uint32_t* d_seed, uint32_t nscalars, uint32_t* d_scalars, char* err, size_t errcap);
  // hash_to_g2 for n seeds (8 words each); d_scalars / d_g2_sx may be null (verification only needs g2_s)
  int (*hash_to_g2)(Ctx& c, int si, uint32_t n, const uint32_t* d_seeds, const uint32_t* d_scalars, uint8_t* d_g2_s, uint8_t* d_g2_sx,
                    char* err, size_t errcap);
  uint32_t fr_words;
  // sum of n uncompressed points -> one uncompressed point (combining per-GPU partial MSM results)
  int (*points_sum)(Ctx& c, int si, uint32_t group, const uint8_t* d_points, uint32_t n, uint8_t* d_out, uint32_t* d_status, char* err, size_t errcap);
  // phase1_cli::new_challenge: n copies of the group generator, uncompressed or compressed
  int (*fill_generator)(Ctx& c, int si, uint32_t group, uint64_t n, uint8_t* d_out, uint32_t out_compressed, char* err, size_t errcap);
  uint32_t fr_bytes;
  uint32_t aff_words[2];     // words per affine point (x|y) in device arrays, per group
  // device time of decoding + checking + the power-ratio MSM of one G2 element relative to one G1 element (measured launch
  // lists, profiles/r2_verify_kernels_*): chunk verification balances its two streams with it
  float verify_g2_weight;
  // radix-2 group FFT of 2^log_n uncompressed points (Stockham stages, natural order in and out; kernels.cuh body_fft_butterfly).
  //   root  : host, canonical words of a root of unity of order 2^two_adicity (its inverse for the inverse transform)
  //   scale : host, canonical Fr bytes multiplying every output (m^-1 of the inverse transform), or null
  // d_out may be d_x; the input is only read.
  int (*group_fft)(Ctx& c, int si, uint32_t group, const uint8_t* d_x, uint32_t log_n, const uint32_t* root, uint32_t two_adicity,
                   const uint8_t* scale, uint8_t* d_out, uint32_t out_compressed, uint32_t* d_status, char* err, size_t errcap);
  // d_out[j] = d_hi[j] - d_lo[j] for n uncompressed points
  int (*points_sub)(Ctx& c, int si, uint32_t group, const uint8_t* d_hi, const uint8_t* d_lo, uint64_t n, uint8_t* d_out,
                    uint32_t out_compressed, char* err, size_t errcap);
  // tau tables (run_tau_tables) for the part twiddle of the four-step group FFT: tau = w^e, w = root^(2^squarings) (root: host,
  // canonical words), first index 0, coefficient slot 0 = scale (host, canonical Fr bytes; null = 1)
  int (*fft_part_tables)(Ctx& c, int si, const uint32_t* root, uint32_t squarings, uint64_t e, const uint8_t* scale, uint32_t** d_table,
                         char* err, size_t errcap);
  // Stockham stage log_ns of the FFT over `rows` rows of row_len uncompressed points (a power of two), natural order in and out:
  // the upper half times w^(row mod 2^log_ns) (w: root^(2^(two_adicity - log_ns - 1)), as in group_fft), then the row butterflies
  // (kernels.cuh body_fft_row_butterfly): d_x -> d_out
  int (*fft_row_stage)(Ctx& c, int si, uint32_t group, const uint8_t* d_x, uint64_t rows, uint64_t row_len, uint32_t log_ns, const uint32_t* root,
                       uint32_t two_adicity, uint32_t* d_status, uint8_t* d_out, char* err, size_t errcap);
};

template <class Fr>
__global__ void k_tau_tables(const uint32_t* tau_canon, const uint32_t* coeff_canon, uint64_t first_index, uint32_t* table) {
  uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
  if (tid < (uint32_t)TAU_TABLE_ELEMS) body_tau_tables<Fr>(tid, tau_canon, coeff_canon, first_index, table);
}

#ifndef SSO_EXP_MIN_BLOCKS
#define SSO_EXP_MIN_BLOCKS 1
#endif
// Resident blocks per SM the register allocation of the single-group kernels aims at, per group (the G1 bodies need far
// fewer registers than the extension-field G2 bodies; a lower register cap buys warps per scheduler to hide the
// fixed-latency dependencies of the carry chains)
#ifndef SSO_EXP_MIN_BLOCKS_G1
#define SSO_EXP_MIN_BLOCKS_G1 SSO_EXP_MIN_BLOCKS
#endif
#ifndef SSO_EXP_MIN_BLOCKS_G2
#define SSO_EXP_MIN_BLOCKS_G2 SSO_EXP_MIN_BLOCKS
#endif
// 1: the two groups of a chunk run as two single-group kernels on two streams (each with its own register budget)
// instead of the one fused launch
#ifndef SSO_SPLIT_GROUPS
#define SSO_SPLIT_GROUPS 0
#endif
template <class G>
__global__ void __launch_bounds__(128, (G::GROUP == 0 ? SSO_EXP_MIN_BLOCKS_G1 : SSO_EXP_MIN_BLOCKS_G2)) k_batch_exp(const __grid_constant__ VecBatch batch, uint32_t in_compressed,
                                                    const uint32_t* table, uint32_t check, uint32_t* jac_out, uint32_t* status) {
  extern __shared__ __align__(16) unsigned char tree_raw[];          // 2 * EXP_BLOCK field elements (dynamic: up to 72 KB)
  block_batch_exp<G>(blockIdx.x, batch, in_compressed, table, check, jac_out, status, reinterpret_cast<typename G::F::T*>(tree_raw));
}

// Every kernel states its resident blocks per SM explicitly: with __launch_bounds__(128) alone ptxas picks the register budget of
// a kernel's whole call tree by an occupancy heuristic and chose 32 registers for the MNT4-753 G2 bucket / fold / window kernels —
// the 24-limb multiplication spilled 7.5 KB per call and k_msm_buckets ran 4.5x slower (profiles/r2_verify_kernels_mnt4_753.txt).
template <class G>
__global__ void __launch_bounds__(128, 1) k_normalize_write(const __grid_constant__ VecBatch batch, const uint32_t* jac,
                                                          uint32_t out_compressed) {
  uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
  body_normalize_write<G>(tid, batch, jac, out_compressed);
}

template <class GC>
__global__ void __launch_bounds__(128, 1) k_subgroup_coop(uint32_t n, const uint32_t* aff, const uint8_t* pts, uint32_t* status) {
  using CO = Coop<GC::F::DEG>;
  if (!CO::lane_active()) return;
  body_subgroup_coop<GC>(blockIdx.x * ExpBlock<GC>::PPB + CO::group_in_block(), n, aff, pts, status);
}

template <class G>
__global__ void __launch_bounds__(128, 1) k_reencode(uint32_t n, const uint8_t* in, uint32_t in_compressed, uint8_t* out,
                                                   uint32_t out_compressed, uint32_t check, uint32_t subgroup, uint32_t* aff_out,
                                                   uint32_t* status) {
  uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
  body_reencode<G>(tid, n, in, in_compressed, out, out_compressed, check, subgroup, aff_out, status);
}

// Both groups of a chunk in ONE launch: blocks [0, nb2) take G2 points (the long-running ones, scheduled first),
// the rest take G1 points.  All blocks have the same register footprint, so G1 blocks fill the SMs that the last,
// partial wave of G2 blocks leaves idle (two separate launches lose ~13 % each to wave quantisation).
#ifndef SSO_CHUNK_MIN_BLOCKS
#define SSO_CHUNK_MIN_BLOCKS 1
#endif
template <class G1, class G2>
__global__ void __launch_bounds__(128, SSO_CHUNK_MIN_BLOCKS) k_batch_exp_chunk(const __grid_constant__ VecBatch b1, const __grid_constant__ VecBatch b2,
                                                          uint32_t nb2, uint32_t in_compressed, const uint32_t* table, uint32_t check,
                                                          uint32_t* jac1, uint32_t* jac2, uint32_t* status) {
  // one dynamic shared buffer, sized by the host for the wider of the two coordinate fields (2 * EXP_BLOCK elements)
  extern __shared__ __align__(16) unsigned char tree_raw[];
  if (blockIdx.x < nb2) {
    block_batch_exp<G2>(blockIdx.x, b2, in_compressed, table, check, jac2, status, reinterpret_cast<typename G2::F::T*>(tree_raw));
  } else {
    block_batch_exp<G1>(blockIdx.x - nb2, b1, in_compressed, table, check, jac1, status, reinterpret_cast<typename G1::F::T*>(tree_raw));
  }
}
template <class G1, class G2>
__global__ void __launch_bounds__(128, 1) k_normalize_chunk(const __grid_constant__ VecBatch b1, const __grid_constant__ VecBatch b2,
                                                          uint32_t nb2, const uint32_t* jac1, const uint32_t* jac2, uint32_t out_compressed) {
  if (blockIdx.x < nb2) body_normalize_write<G2>(blockIdx.x * blockDim.x + threadIdx.x, b2, jac2, out_compressed);
  else body_normalize_write<G1>((blockIdx.x - nb2) * blockDim.x + threadIdx.x, b1, jac1, out_compressed);
}

// The extension-field groups run their batch_exp bodies warp-cooperatively (coop.cuh: one coefficient per lane) on uncompressed
// input; SSO_COOP_G2=0 in the environment selects the one-thread-per-element bodies (A/B measurements, tools/).
// Default per curve (measured on B200, profiles/r2_coop_ab.txt): on for the 753-bit towers, off for BLS12-377 (12-limb
// coefficients: four base multiplications per Fq2 product instead of Karatsuba's three cost more than the registers gain).
//   -1 = not set, 0 / 1 = forced
inline int coop_g2_override() {
  const char* e = getenv("SSO_COOP_G2");                // read per call: the parity tests run both bodies in one process
  return !e || !e[0] ? -1 : (e[0] == '0' ? 0 : 1);
}
template <class GC> inline bool coop_g2_enabled() {
  int o = coop_g2_override();
  return o < 0 ? GC::COOP_DEFAULT : o != 0;
}

template <class G1, class G2>
inline int run_batch_exp_chunk(Ctx& c, int si, const VecBatch& b1, const VecBatch& b2, uint32_t in_compressed, const uint32_t* d_table,
                               uint32_t out_compressed, uint32_t check, uint32_t* d_status, char* err, size_t errcap) {
  uint64_t n1 = b1.total, n2 = b2.total;
  if (n1 + n2 == 0) return SSO_OK;
  for (uint32_t i = 0; i < b1.nseg; i++) if (b1.seg[i].n > (1u << 24)) { set_err(err, errcap, "vector longer than 2^24 elements: split the call"); return SSO_E_ARG; }
  for (uint32_t i = 0; i < b2.nseg; i++) if (b2.seg[i].n > (1u << 24)) { set_err(err, errcap, "vector longer than 2^24 elements: split the call"); return SSO_E_ARG; }
  cudaStream_t st = c.s[si];
  uint32_t *d_jac1 = nullptr, *d_jac2 = nullptr;
  int rc;
  if ((rc = c.alloc((void**)&d_jac1, (size_t)n1 * 3 * G1::F::WORDS * 4, si))) return rc;
  if ((rc = c.alloc((void**)&d_jac2, (size_t)n2 * 3 * G2::F::WORDS * 4, si))) return rc;
  uint32_t nb2 = div_up(n2, EXP_BLOCK), nb1 = div_up(n1, EXP_BLOCK);
  constexpr size_t TREE_BYTES = 16 + 2 * EXP_BLOCK * (sizeof(typename G1::F::T) > sizeof(typename G2::F::T) ? sizeof(typename G1::F::T)
                                                                                                             : sizeof(typename G2::F::T));
  // per device and cheap: set on every call (a process-wide "done" flag would leave the other GPUs of the box unset)
  if (TREE_BYTES > 48 * 1024)
    CUDA_TRY(cudaFuncSetAttribute(k_batch_exp_chunk<G1, G2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TREE_BYTES));
#if SSO_SPLIT_GROUPS
  {
    // G2 (the longer blocks) on the call's stream, G1 beside it on the second stream; both drain before the normalisation
    const int sj = (c.s[1] && !c.aliased) ? 1 : si;
    constexpr size_t TREE1 = 16 + 2 * EXP_BLOCK * sizeof(typename G1::F::T), TREE2 = 16 + 2 * EXP_BLOCK * sizeof(typename G2::F::T);
    if (TREE1 > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(k_batch_exp<G1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TREE1));
    if (TREE2 > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(k_batch_exp<G2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TREE2));
    if (sj != si && (rc = c.fork(si, sj))) return rc;
    if (n2) {
      c.begin(PK_BATCH_EXP_G2, si, n2);
      k_batch_exp<G2><<<nb2, EXP_BLOCK, TREE2, st>>>(b2, in_compressed, d_table, check, d_jac2, d_status);
      c.end(si);
    }
    if (n1) {
      c.begin(PK_BATCH_EXP_G1, sj, n1);
      k_batch_exp<G1><<<nb1, EXP_BLOCK, TREE1, c.s[sj]>>>(b1, in_compressed, d_table, check, d_jac1, d_status);
      c.end(sj);
    }
    if (sj != si && (rc = c.fork(sj, si))) return rc;
  }
#else
  using G2C = typename CoopOf<G2>::type;
  bool coop = false;
  if constexpr (!std::is_void<G2C>::value) {
    if (!in_compressed && coop_g2_enabled<G2C>()) {
      coop = true;
      constexpr size_t SM1 = 16 + 2 * EXP_BLOCK * sizeof(typename G1::F::T);
      constexpr size_t SMEM = SM1 > ExpBlock<G2C>::SMEM ? SM1 : ExpBlock<G2C>::SMEM;
      if (SMEM > 48 * 1024)
        CUDA_TRY(cudaFuncSetAttribute(k_batch_exp_chunk<G1, G2C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
      nb2 = div_up(n2, ExpBlock<G2C>::PPB);
      c.begin(PK_BATCH_EXP_CHUNK, si, n1 + n2);
      k_batch_exp_chunk<G1, G2C><<<nb1 + nb2, EXP_BLOCK, SMEM, st>>>(b1, b2, nb2, 0, d_table, check, d_jac1, d_jac2, d_status);
      c.end(si);
    }
  }
  if (!coop) {
    c.begin(PK_BATCH_EXP_CHUNK, si, n1 + n2);
    k_batch_exp_chunk<G1, G2><<<nb1 + nb2, EXP_BLOCK, TREE_BYTES, st>>>(b1, b2, nb2, in_compressed, d_table, check, d_jac1, d_jac2, d_status);
    c.end(si);
  }
#endif
  uint32_t mb2 = div_up(div_up(n2, NORM_BATCH), 128), mb1 = div_up(div_up(n1, NORM_BATCH), 128);
  c.begin(PK_NORMALIZE_CHUNK, si, n1 + n2);
  k_normalize_chunk<G1, G2><<<mb1 + mb2, 128, 0, st>>>(b1, b2, mb2, d_jac1, d_jac2, out_compressed);
  c.end(si);
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

// tau tables for one call: powers of tau from first_index plus up to three coefficient slots
template <class Fr>
inline int run_tau_tables(Ctx& c, int si, uint64_t first_index, const uint8_t* tau, const uint8_t* const coeffs[TAU_COEFF_SLOTS],
                          uint32_t** d_table, char* err, size_t errcap) {
  c.staging.emplace_back((size_t)(1 + TAU_COEFF_SLOTS) * Fr::L, 0u);
  std::vector<uint32_t>& w = c.staging.back();
  if (tau) memcpy(w.data(), tau, Fr::NBYTES); else w[0] = 1;
  for (int i = 0; i < TAU_COEFF_SLOTS; i++) {
    if (coeffs && coeffs[i]) memcpy(w.data() + (size_t)(1 + i) * Fr::L, coeffs[i], Fr::NBYTES);
    else w[(size_t)(1 + i) * Fr::L] = 1;
  }
  uint32_t* d_sc;
  int rc;
  if ((rc = c.alloc((void**)&d_sc, w.size() * 4, si))) return rc;
  if ((rc = c.alloc((void**)d_table, (size_t)TAU_TABLE_ELEMS * Fr::L * 4, si))) return rc;
  CUDA_TRY(cudaMemcpyAsync(d_sc, w.data(), w.size() * 4, cudaMemcpyHostToDevice, c.s[si]));
  c.begin(PK_TAU_TABLES, si, TAU_TABLE_ELEMS);
  k_tau_tables<Fr><<<div_up(TAU_TABLE_ELEMS, 128), 128, 0, c.s[si]>>>(d_sc, d_sc + Fr::L, first_index, *d_table);
  c.end(si);
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

// K2-K4 for up to four vectors of one group in ONE launch pair (batch_exp + normalize) on stream si
template <class G>
inline int run_batch_exp(Ctx& c, int si, const VecBatch& batch, uint32_t in_compressed, const uint32_t* d_table,
                         uint32_t out_compressed, uint32_t check, uint32_t* d_status, char* err, size_t errcap) {
  using F = typename G::F;
  uint64_t n = batch.total;
  if (n == 0) return SSO_OK;
  for (uint32_t i = 0; i < batch.nseg; i++)
    if (batch.seg[i].n > (1u << 24)) { set_err(err, errcap, "vector longer than 2^24 elements: split the call"); return SSO_E_ARG; }
  cudaStream_t st = c.s[si];
  uint32_t* d_jac = nullptr;
  int rc;
  if ((rc = c.alloc((void**)&d_jac, (size_t)n * 3 * F::WORDS * 4, si))) return rc;
  constexpr bool IS_G1 = G::GROUP == 0;
  constexpr size_t TREE_BYTES = 16 + 2 * EXP_BLOCK * sizeof(typename F::T);
  if (TREE_BYTES > 48 * 1024)
    CUDA_TRY(cudaFuncSetAttribute(k_batch_exp<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TREE_BYTES));
  using GC = typename CoopOf<G>::type;
  bool coop = false;
  if constexpr (!std::is_void<GC>::value) {
    if (!in_compressed && coop_g2_enabled<GC>()) {
      coop = true;
      if (ExpBlock<GC>::SMEM > 48 * 1024)
        CUDA_TRY(cudaFuncSetAttribute(k_batch_exp<GC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ExpBlock<GC>::SMEM));
      c.begin(PK_BATCH_EXP_G2, si, n);
      k_batch_exp<GC><<<div_up(n, ExpBlock<GC>::PPB), EXP_BLOCK, ExpBlock<GC>::SMEM, st>>>(batch, 0, d_table, check, d_jac, d_status);
      c.end(si);
    }
  }
  if (!coop) {
    c.begin(IS_G1 ? PK_BATCH_EXP_G1 : PK_BATCH_EXP_G2, si, n);
    k_batch_exp<G><<<div_up(n, EXP_BLOCK), EXP_BLOCK, TREE_BYTES, st>>>(batch, in_compressed, d_table, check, d_jac, d_status);
    c.end(si);
  }
  c.begin(IS_G1 ? PK_NORMALIZE_G1 : PK_NORMALIZE_G2, si, n);
  k_normalize_write<G><<<div_up(div_up(n, NORM_BATCH), 128), 128, 0, st>>>(batch, d_jac, out_compressed);
  c.end(si);
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

template <class G>
__global__ void k_fill_generator(uint32_t n, uint8_t* out, uint32_t out_compressed) {
  using C = SW<G>;
  uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= n) return;
  typename C::Affine g{G::gen_x(), G::gen_y(), false};
  if (out_compressed) C::write_compressed(out + (size_t)tid * C::SIZE_C, g);
  else C::write_uncompressed(out + (size_t)tid * C::SIZE_U, g);
}

template <class G>
inline int run_fill_generator(Ctx& c, int si, uint64_t n, uint8_t* d_out, uint32_t out_compressed, char* err, size_t errcap) {
  if (n == 0) return SSO_OK;
  if (n > 0xffffffffull) { set_err(err, errcap, "vector too long"); return SSO_E_ARG; }
  c.begin(PK_FILL, si, n);
  k_fill_generator<G><<<div_up(n, 128), 128, 0, c.s[si]>>>((uint32_t)n, d_out, out_compressed);
  c.end(si);
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

// the ChaCha20 key travels as a kernel argument: a pageable-memory cudaMemcpyAsync would make the host wait for the
// kernels already queued on the stream (measured: 120 ms of lost overlap per chunk verification)
struct Key32 { uint32_t w[8]; };
template <class G>
__global__ void k_random_scalars(uint32_t n, const __grid_constant__ Key32 key, uint32_t* scalars) {
  body_random_scalars<RLC_WORDS, RLC_BITS>(blockIdx.x * blockDim.x + threadIdx.x, n, key.w, scalars);
}
template <class G>
__global__ void k_msm_keys(uint32_t n, uint32_t nwin, uint32_t c, const uint32_t* scalars, uint32_t* keys, uint32_t* vals) {
  body_msm_keys<RLC_WORDS>(blockIdx.x * blockDim.x + threadIdx.x, n, nwin, c, scalars, keys, vals);
}
template <class G>
__global__ void __launch_bounds__(128, 1) k_msm_buckets(uint32_t n, uint32_t nwin, uint32_t c, const uint32_t* keys, const uint32_t* vals,
                                                      const uint32_t* aff_a, const uint32_t* aff_b, uint32_t* buckets) {
  body_msm_buckets<G>(blockIdx.x * blockDim.x + threadIdx.x, n, nwin, c, keys, vals, aff_a, aff_b, buckets);
}
template <class G>
__global__ void __launch_bounds__(128, 1) k_msm_fold(uint32_t nwin, uint32_t c, const uint32_t* buckets, uint32_t* seg_out) {
  body_msm_fold<G>(blockIdx.x * blockDim.x + threadIdx.x, nwin, c, buckets, seg_out);
}
template <class G>
__global__ void __launch_bounds__(128, 1) k_msm_window(uint32_t nwin, uint32_t c, const uint32_t* seg_in, uint32_t* win_out) {
  body_msm_window<G>(blockIdx.x * blockDim.x + threadIdx.x, nwin, c, seg_in, win_out);
}
template <class G>
__global__ void __launch_bounds__(128, 1) k_msm_final(uint32_t nwin, uint32_t c, const uint32_t* win_in, uint8_t* out) {
  body_msm_final<G>(blockIdx.x * blockDim.x + threadIdx.x, nwin, c, win_in, out);
}

template <class G1, class G2, class PP>
__global__ void __launch_bounds__(64, 1) k_same_ratio(const uint8_t* checks, uint32_t* verdicts) {
  using PR = Pairing<G1, G2, PP>;
  using Fq = typename G1::F;
  __shared__ typename PR::Ws ws[2];
  __shared__ uint32_t st[2];
  int side = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t s = PR::run_side(lane, ws[side], checks + (size_t)blockIdx.x * PR::CHECK_BYTES, side);
  if (lane == 0) st[side] = s;
  __syncthreads();
  if (side == 0) {
    bool bad = (st[0] | st[1]) != 0;
    bool ok = false;
    if (!bad) ok = PR::combine_and_check(lane, ws[0], ws[1]);      // one final exponentiation for the pair of Miller values
    if (lane == 0) verdicts[blockIdx.x] = bad ? 0x100u + (st[0] ? st[0] : st[1]) : (ok ? 1u : 0u);
  }
}

template <class G1, class G2, class PP>
inline int run_same_ratio(Ctx& c, int si, const uint8_t* d_checks, uint64_t n, uint32_t* d_verdicts, char* err, size_t errcap) {
  if (n == 0) return SSO_OK;
  if (n > 65535) { set_err(err, errcap, "too many same_ratio checks in one call"); return SSO_E_ARG; }
  c.begin(PK_OTHER, si, n);
  k_same_ratio<G1, G2, PP><<<(uint32_t)n, 64, 0, c.s[si]>>>(d_checks, d_verdicts);
  c.end(si);
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

template <class G1>
__global__ void k_keygen_g1(const uint32_t* seed, uint32_t nscalars, uint32_t* scalars_out, uint8_t* g1_out) {
  // thread 0 draws from the RNG; then the first lane of warp i finishes proof i (cofactor clearing, [x]s): the three long
  // single-thread chains run side by side instead of one after the other
  __shared__ typename SW<G1>::Affine raw[3];
  if (threadIdx.x == 0) keygen_g1_sample<G1>(seed, nscalars, scalars_out, raw);
  __syncthreads();
  uint32_t i = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0 && i < nscalars) keygen_g1_finish<G1>(i, raw[i], scalars_out, g1_out);
}
template <class G1>
__global__ void k_keygen_scalars(const uint32_t* seed, uint32_t nscalars, uint32_t* scalars_out) {
  using Fr = typename G1::Fr;
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  ChaChaStream rng;
  rng.init(seed);
  for (uint32_t i = 0; i < nscalars; i++) {
    typename Fr::T c = Fr::from_mont(fp_rand<Fr>(rng));
    for (int w = 0; w < Fr::L; w++) scalars_out[i * Fr::L + w] = c.v[w];
  }
}
template <class G2>
__global__ void k_hash_to_g2(uint32_t n, const uint32_t* seeds, const uint32_t* scalars, uint8_t* g2_s, uint8_t* g2_sx) {
  // one point per block so that the long single-thread chains land on different SMs
  if (threadIdx.x == 0) body_hash_to_g2<G2>(blockIdx.x, n, seeds, scalars, g2_s, g2_sx);
}

template <class G>
__global__ void k_points_sum(const uint8_t* pts, uint32_t n, uint8_t* out, uint32_t* status) {
  using C = SW<G>;
  using F = typename G::F;
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  typename C::Jac acc = C::identity();
  for (uint32_t i = 0; i < n; i++) {
    typename C::Affine p;
    uint32_t st = C::read_uncompressed(pts + (size_t)i * C::SIZE_U, p);
    if (st != C::DESER_OK || !C::on_curve(p)) { report(status, st ? st : (uint32_t)ST_NOT_ON_CURVE, i); return; }
    acc = C::madd(acc, p);
  }
  C::write_uncompressed(out, jac_to_affine<G>(acc));
}
template <class G>
inline int run_points_sum(Ctx& c, int si, const uint8_t* d_points, uint32_t n, uint8_t* d_out, uint32_t* d_status, char* err, size_t errcap) {
  c.begin(PK_OTHER, si, n);
  k_points_sum<G><<<1, 32, 0, c.s[si]>>>(d_points, n, d_out, d_status);
  c.end(si);
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

// Window width of the Pippenger MSM.  One thread sums one bucket, so the bucket phase lasts as long as the longest bucket
// (n >> c points when every window is full); the fold adds 2 * MSM_SEG points per thread and the window stage walks the
// 2^c / MSM_SEG segments of a window serially.  Among the widths that divide the scalar length (no partial top window)
// pick the one with the shortest chain of dependent point additions (mixed addition ~ 11, full addition ~ 16 multiplications).
inline uint32_t msm_window_bits(uint64_t n, uint32_t sbits) {
  static const uint32_t cands[] = {4, 5, 6, 8, 10, 12};
  uint32_t best = 4;
  uint64_t best_cost = ~0ull;
  for (uint32_t c : cands) {
    if (sbits % c) continue;
    uint64_t nb = 1ull << c, seg = nb < MSM_SEG ? nb : MSM_SEG;
    uint64_t cost = (n >> c) * 11 + 2 * seg * 16 + 3 * (nb / seg) * 16;
    if (cost < best_cost) { best_cost = cost; best = c; }
  }
  return best;
}

template <class G>
inline int run_msm_pairs(Ctx& c, int si, const uint32_t* d_aff_a, const uint32_t* d_aff_b, uint64_t n, const uint8_t seed32[32],
                         const uint64_t* tweak, uint8_t* d_out, char* err, size_t errcap) {
  using F = typename G::F;
  using Fr = typename G::Fr;
  constexpr int KL = RLC_WORDS;
  constexpr int SBITS = RLC_BITS;
  static_assert(RLC_BITS < Fr::P::BITS, "the random scalars must stay below the group order");
  if (n == 0 || n > (1ull << 26)) { set_err(err, errcap, "msm length out of range"); return SSO_E_ARG; }
  cudaStream_t st = c.s[si];
  uint32_t wb = msm_window_bits(n, SBITS), nwin = (SBITS + wb - 1) / wb, nb = 1u << wb;
  uint32_t seg = nb < MSM_SEG ? nb : MSM_SEG, nseg = nb / seg;
  size_t pairs = (size_t)n * nwin;
  if (pairs > 0x7fffffffull) { set_err(err, errcap, "msm too large for 32-bit indexing (cub takes an int count): split the vector"); return SSO_E_ARG; }
  // scalar key: fresh host entropy, or — reproducible runs, tests — derived from the caller's seed and the tweak that
  // names this MSM (vector, chunk, piece offset, rank): two MSMs with the same r_i would make the G1-vs-G2 power-ratio
  // check vacuous for correlated vectors
  Key32 key;
  if (seed32 && tweak) {
    Blake2b h(32);
    h.update(seed32, 32);
    h.update((const uint8_t*)tweak, 32);
    h.final((uint8_t*)key.w, 32);
  } else if (seed32) memcpy(key.w, seed32, 32);
  else { std::random_device rd; for (auto& w : key.w) w = rd(); }
  uint32_t *d_sc, *d_keys, *d_vals, *d_keys2, *d_vals2, *d_buckets, *d_seg, *d_win;
  void* d_tmp = nullptr;
  int rc;
  if ((rc = c.alloc((void**)&d_sc, (size_t)n * KL * 4, si))) return rc;
  if ((rc = c.alloc((void**)&d_keys, pairs * 4, si))) return rc;
  if ((rc = c.alloc((void**)&d_vals, pairs * 4, si))) return rc;
  if ((rc = c.alloc((void**)&d_keys2, pairs * 4, si))) return rc;
  if ((rc = c.alloc((void**)&d_vals2, pairs * 4, si))) return rc;
  if ((rc = c.alloc((void**)&d_buckets, (size_t)2 * nwin * nb * 3 * F::WORDS * 4, si))) return rc;
  if ((rc = c.alloc((void**)&d_seg, (size_t)2 * nwin * nseg * 6 * F::WORDS * 4, si))) return rc;
  if ((rc = c.alloc((void**)&d_win, (size_t)2 * nwin * 3 * F::WORDS * 4, si))) return rc;
  size_t tmp_bytes = 0;
  uint32_t key_bits = wb;
  while ((1u << (key_bits - wb)) < nwin) key_bits++;
  CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, d_keys, d_keys2, d_vals, d_vals2, (int)pairs, 0, (int)key_bits, st));
  if ((rc = c.alloc(&d_tmp, tmp_bytes, si))) return rc;
  c.begin(PK_MSM, si, n);
  k_random_scalars<G><<<div_up(n, 128), 128, 0, st>>>((uint32_t)n, key, d_sc);
  k_msm_keys<G><<<div_up(n, 128), 128, 0, st>>>((uint32_t)n, nwin, wb, d_sc, d_keys, d_vals);
  CUDA_TRY(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, d_keys, d_keys2, d_vals, d_vals2, (int)pairs, 0, (int)key_bits, st));
  k_msm_buckets<G><<<div_up((uint64_t)nwin * nb, 128), 128, 0, st>>>((uint32_t)n, nwin, wb, d_keys2, d_vals2, d_aff_a, d_aff_b, d_buckets);
  k_msm_fold<G><<<div_up((uint64_t)2 * nwin * nseg, 128), 128, 0, st>>>(nwin, wb, d_buckets, d_seg);
  k_msm_window<G><<<div_up((uint64_t)2 * nwin, 128), 128, 0, st>>>(nwin, wb, d_seg, d_win);
  k_msm_final<G><<<1, 32, 0, st>>>(nwin, wb, d_win, d_out);
  c.end(si);
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

template <class G>
inline int run_reencode(Ctx& c, int si, const uint8_t* d_in, uint32_t in_compressed, uint64_t n, uint8_t* d_out,
                        uint32_t out_compressed, uint32_t check, uint32_t subgroup, uint32_t* d_aff, uint32_t* d_status,
                        char* err, size_t errcap) {
  if (n == 0) return SSO_OK;
  if (n > 0xffffffffull) { set_err(err, errcap, "vector too long"); return SSO_E_ARG; }
  constexpr bool IS_G1 = G::GROUP == 0;
  // the membership test of the 753-bit extension-field groups runs through the cooperative fields (2 / 3 lanes per point) in a
  // second kernel over the decoded points; SSO_COOP_G2 = 0 keeps it inside the decoding kernel
  using GC = typename CoopOf<G>::type;
  bool coop = false;
  if constexpr (!std::is_void<GC>::value) {
    if constexpr (GC::ENDO_SUBGROUP_TEST == 4)
      coop = subgroup && (d_aff || (d_out && !out_compressed)) && coop_g2_enabled<GC>();
  }
  c.begin(IS_G1 ? PK_REENCODE_G1 : PK_REENCODE_G2, si, n);
  k_reencode<G><<<div_up(n, 128), 128, 0, c.s[si]>>>((uint32_t)n, d_in, in_compressed, d_out, out_compressed, check, coop ? 2u : subgroup, d_aff, d_status);
  if constexpr (!std::is_void<GC>::value) {
    if (coop) k_subgroup_coop<GC><<<div_up(n, ExpBlock<GC>::PPB), 128, 0, c.s[si]>>>((uint32_t)n, d_aff, d_aff ? nullptr : d_out, d_status);
  }
  c.end(si);
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

// ---------------------------------------------------------------------------------------------
// group FFT (prepare_phase2)
// ---------------------------------------------------------------------------------------------
// the root of unity of one Stockham stage, root^(2^squarings), canonical, followed by three canonical ones: the input of
// k_tau_tables (tau + coefficient slots)
template <class Fr>
__global__ void __launch_bounds__(128, 1) k_fft_stage_root(const uint32_t* root_canon, uint32_t squarings, uint32_t* out_canon) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  typename Fr::T w = Fr::to_mont(Fr::from_const(root_canon));
  for (uint32_t i = 0; i < squarings; i++) w = Fr::sqr(w);
  w = Fr::from_mont(w);
  for (int i = 0; i < Fr::L; i++) out_canon[i] = w.v[i];
  for (int k = 1; k <= TAU_COEFF_SLOTS; k++)
    for (int i = 0; i < Fr::L; i++) out_canon[k * Fr::L + i] = i == 0 ? 1u : 0u;
}
// t_j = w^(j & tw_mask) x[j] over one segment: the batch_exp body with the twiddle scalar source (a separate instantiation,
// so the k_batch_exp code is unchanged)
template <class G>
__global__ void __launch_bounds__(128, (G::GROUP == 0 ? SSO_EXP_MIN_BLOCKS_G1 : SSO_EXP_MIN_BLOCKS_G2)) k_fft_twiddle(const __grid_constant__ VecBatch batch,
                                                    const uint32_t* table, uint32_t tw_mask, uint32_t* jac_out, uint32_t* status) {
  extern __shared__ __align__(16) unsigned char tree_raw[];
  block_batch_exp<G, true>(blockIdx.x, batch, 0, table, CHECK_NO, jac_out, status, reinterpret_cast<typename G::F::T*>(tree_raw), tw_mask);
}
template <class G>
__global__ void __launch_bounds__(128, 1) k_fft_butterfly(uint32_t half, uint32_t log_ns, const uint8_t* x, const uint32_t* tw, uint32_t* jac_out) {
  body_fft_butterfly<G>(blockIdx.x * blockDim.x + threadIdx.x, half, log_ns, x, tw, jac_out);
}
template <class G>
__global__ void __launch_bounds__(128, 1) k_points_sub(uint32_t n, const uint8_t* hi, const uint8_t* lo, uint32_t* jac_out) {
  body_points_sub<G>(blockIdx.x * blockDim.x + threadIdx.x, n, hi, lo, jac_out);
}

template <class G>
inline int run_normalize_other(Ctx& c, int si, const uint32_t* d_jac, uint64_t n, uint8_t* d_out, uint32_t out_compressed) {
  VecBatch o;
  memset(&o, 0, sizeof o);
  o.seg[0].out = d_out; o.seg[0].n = (uint32_t)n; o.nseg = 1; o.total = (uint32_t)n;
  c.begin(PK_OTHER, si, n);
  k_normalize_write<G><<<div_up(div_up(n, NORM_BATCH), 128), 128, 0, c.s[si]>>>(o, d_jac, out_compressed);
  c.end(si);
  return SSO_OK;
}

template <class G>
inline int run_group_fft(Ctx& c, int si, const uint8_t* d_x, uint32_t log_n, const uint32_t* root, uint32_t two_adicity, const uint8_t* scale,
                         uint8_t* d_out, uint32_t out_compressed, uint32_t* d_status, char* err, size_t errcap) {
  using F = typename G::F;
  using Fr = typename G::Fr;
  using C = SW<G>;
  if (log_n > two_adicity || log_n > 24) { set_err(err, errcap, "group FFT of 2^%u points: beyond the radix-2 domain (2^%u) or 2^24", log_n, two_adicity < 24 ? two_adicity : 24); return SSO_E_ARG; }
  const uint64_t n = 1ull << log_n, half = n / 2;
  cudaStream_t st = c.s[si];
  int rc;
  const uint8_t* cur = d_x;
  uint8_t* buf[2] = {nullptr, nullptr};
  if (log_n > 0)
    for (auto& b : buf) if ((rc = c.alloc((void**)&b, n * C::SIZE_U, si))) return rc;
  if (scale) {
    // x * m^-1: one shared-scalar pass before the stages (the a-path of a butterfly has no multiplication to fold it into)
    const uint8_t* coeffs[TAU_COEFF_SLOTS] = {scale, nullptr, nullptr};
    uint32_t* d_table;
    if ((rc = run_tau_tables<Fr>(c, si, 0, nullptr, coeffs, &d_table, err, errcap))) return rc;
    VecBatch b;
    memset(&b, 0, sizeof b);
    b.seg[0].in = d_x; b.seg[0].out = log_n ? buf[0] : d_out; b.seg[0].n = (uint32_t)n; b.seg[0].has_coeff = 1; b.seg[0].mode = 1;
    b.nseg = 1; b.total = (uint32_t)n;
    if ((rc = run_batch_exp<G>(c, si, b, 0, d_table, log_n ? 0 : out_compressed, CHECK_NO, d_status, err, errcap))) return rc;
    if (log_n == 0) return SSO_OK;
    cur = buf[0];
  } else if (log_n == 0) {
    return run_reencode<G>(c, si, d_x, 0, 1, d_out, out_compressed, CHECK_NO, 0, nullptr, d_status, err, errcap);
  }
  uint32_t *d_root, *d_stage, *d_table, *d_jac, *d_tw;
  if ((rc = upload_scalar(c, (const uint8_t*)root, (size_t)Fr::L * 4, Fr::L, &d_root, si, err, errcap))) return rc;
  if ((rc = c.alloc((void**)&d_stage, (size_t)(1 + TAU_COEFF_SLOTS) * Fr::L * 4, si))) return rc;
  if ((rc = c.alloc((void**)&d_table, (size_t)TAU_TABLE_ELEMS * Fr::L * 4, si))) return rc;
  if ((rc = c.alloc((void**)&d_jac, n * 3 * F::WORDS * 4, si))) return rc;
  if ((rc = c.alloc((void**)&d_tw, half * 3 * F::WORDS * 4, si))) return rc;
  using GC = typename CoopOf<G>::type;
  bool coop = false;
  if constexpr (!std::is_void<GC>::value) coop = coop_g2_enabled<GC>();
  constexpr size_t TREE_BYTES = 16 + 2 * EXP_BLOCK * sizeof(typename F::T);
  if (TREE_BYTES > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(k_fft_twiddle<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TREE_BYTES));
  for (uint32_t s = 0; s < log_n; s++) {
    uint8_t* nxt = s + 1 == log_n ? d_out : (cur == buf[0] ? buf[1] : buf[0]);
    const uint32_t* tw = nullptr;
    if (s > 0) {
      // twiddles of stage s: powers of the root of order 2^(s+1), for the upper half x[n/2 ..)
      c.begin(PK_OTHER, si, TAU_TABLE_ELEMS);
      k_fft_stage_root<Fr><<<1, 32, 0, st>>>(d_root, two_adicity - (s + 1), d_stage);
      k_tau_tables<Fr><<<div_up(TAU_TABLE_ELEMS, 128), 128, 0, st>>>(d_stage, d_stage + Fr::L, 0, d_table);
      c.end(si);
      VecBatch b;
      memset(&b, 0, sizeof b);
      b.seg[0].in = cur + half * C::SIZE_U; b.seg[0].n = (uint32_t)half; b.nseg = 1; b.total = (uint32_t)half;
      const uint32_t mask = (1u << s) - 1;
      c.begin(G::GROUP == 0 ? PK_BATCH_EXP_G1 : PK_BATCH_EXP_G2, si, half);
      if constexpr (!std::is_void<GC>::value) {
        if (coop) {
          if (ExpBlock<GC>::SMEM > 48 * 1024)
            CUDA_TRY(cudaFuncSetAttribute(k_fft_twiddle<GC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ExpBlock<GC>::SMEM));
          k_fft_twiddle<GC><<<div_up(half, ExpBlock<GC>::PPB), EXP_BLOCK, ExpBlock<GC>::SMEM, st>>>(b, d_table, mask, d_tw, d_status);
        }
      }
      if (!coop) k_fft_twiddle<G><<<div_up(half, EXP_BLOCK), EXP_BLOCK, TREE_BYTES, st>>>(b, d_table, mask, d_tw, d_status);
      c.end(si);
      tw = d_tw;
    }
    c.begin(PK_OTHER, si, n);
    k_fft_butterfly<G><<<div_up(half, 128), 128, 0, st>>>((uint32_t)half, s, cur, tw, d_jac);
    c.end(si);
    run_normalize_other<G>(c, si, d_jac, n, nxt, s + 1 == log_n ? out_compressed : 0);
    cur = nxt;
  }
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

// the input of k_tau_tables for the part twiddle of the four-step group FFT: tau = w^e with w = root^(2^squarings), then the
// coefficient slots scale (canonical; null = 1), 1, 1
template <class Fr>
__global__ void __launch_bounds__(128, 1) k_fft_part_root(const uint32_t* root_canon, uint32_t squarings, uint64_t e, const uint32_t* scale_canon,
                                                        uint32_t* out_canon) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  typename Fr::T w = Fr::to_mont(Fr::from_const(root_canon));
  for (uint32_t i = 0; i < squarings; i++) w = Fr::sqr(w);
  w = Fr::from_mont(fr_pow_u64<Fr>(w, e));
  for (int i = 0; i < Fr::L; i++) out_canon[i] = w.v[i];
  for (int k = 1; k <= TAU_COEFF_SLOTS; k++)
    for (int i = 0; i < Fr::L; i++) out_canon[k * Fr::L + i] = k == 1 && scale_canon ? scale_canon[i] : (i == 0 ? 1u : 0u);
}
// t_e = w^((e >> row_shift) & tw_mask) x[e]: the twiddles of the FFT over rows of 2^row_shift points (the row index as exponent)
template <class G>
__global__ void __launch_bounds__(128, (G::GROUP == 0 ? SSO_EXP_MIN_BLOCKS_G1 : SSO_EXP_MIN_BLOCKS_G2)) k_fft_row_twiddle(const __grid_constant__ VecBatch batch,
                                                    const uint32_t* table, uint32_t tw_mask, uint32_t row_shift, uint32_t* jac_out, uint32_t* status) {
  extern __shared__ __align__(16) unsigned char tree_raw[];
  block_batch_exp<G, true>(blockIdx.x, batch, 0, table, CHECK_NO, jac_out, status, reinterpret_cast<typename G::F::T*>(tree_raw), tw_mask, row_shift);
}
template <class G>
__global__ void __launch_bounds__(128, 1) k_fft_row_butterfly(uint32_t half, uint32_t row_len, uint32_t log_ns, const uint8_t* x, const uint32_t* tw,
                                                            uint32_t* jac_out) {
  body_fft_row_butterfly<G>(blockIdx.x * blockDim.x + threadIdx.x, half, row_len, log_ns, x, tw, jac_out);
}

template <class Fr>
inline int run_fft_part_tables(Ctx& c, int si, const uint32_t* root, uint32_t squarings, uint64_t e, const uint8_t* scale, uint32_t** d_table,
                               char* err, size_t errcap) {
  uint32_t *d_root, *d_scale = nullptr, *d_sc;
  int rc;
  if ((rc = upload_scalar(c, (const uint8_t*)root, (size_t)Fr::L * 4, Fr::L, &d_root, si, err, errcap))) return rc;
  if (scale && (rc = upload_scalar(c, scale, Fr::NBYTES, Fr::L, &d_scale, si, err, errcap))) return rc;
  if ((rc = c.alloc((void**)&d_sc, (size_t)(1 + TAU_COEFF_SLOTS) * Fr::L * 4, si))) return rc;
  if ((rc = c.alloc((void**)d_table, (size_t)TAU_TABLE_ELEMS * Fr::L * 4, si))) return rc;
  c.begin(PK_TAU_TABLES, si, TAU_TABLE_ELEMS);
  k_fft_part_root<Fr><<<1, 32, 0, c.s[si]>>>(d_root, squarings, e, d_scale, d_sc);
  k_tau_tables<Fr><<<div_up(TAU_TABLE_ELEMS, 128), 128, 0, c.s[si]>>>(d_sc, d_sc + Fr::L, 0, *d_table);
  c.end(si);
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

// Stage log_ns of the FFT over `rows` rows of row_len points (a power of two): the twiddles of the upper half (one launch, the row
// index as exponent of the stage root), then the row butterflies into Jacobian scratch and their normalisation into d_out
template <class G>
inline int run_fft_row_stage(Ctx& c, int si, const uint8_t* d_x, uint64_t rows, uint64_t row_len, uint32_t log_ns, const uint32_t* root,
                             uint32_t two_adicity, uint32_t* d_status, uint8_t* d_out, char* err, size_t errcap) {
  using F = typename G::F;
  using Fr = typename G::Fr;
  using C = SW<G>;
  const uint64_t n = rows * row_len, half = n / 2;
  if (rows < 2 || n > (1ull << 24) || (row_len & (row_len - 1))) {
    set_err(err, errcap, "row FFT stage of %llu x %llu points", (unsigned long long)rows, (unsigned long long)row_len);
    return SSO_E_ARG;
  }
  cudaStream_t st = c.s[si];
  uint32_t *d_jac, *d_tw = nullptr;
  int rc;
  if ((rc = c.alloc((void**)&d_jac, n * 3 * F::WORDS * 4, si))) return rc;
  if (log_ns > 0) {
    uint32_t *d_root, *d_stage, *d_table;
    if ((rc = upload_scalar(c, (const uint8_t*)root, (size_t)Fr::L * 4, Fr::L, &d_root, si, err, errcap))) return rc;
    if ((rc = c.alloc((void**)&d_stage, (size_t)(1 + TAU_COEFF_SLOTS) * Fr::L * 4, si))) return rc;
    if ((rc = c.alloc((void**)&d_table, (size_t)TAU_TABLE_ELEMS * Fr::L * 4, si))) return rc;
    if ((rc = c.alloc((void**)&d_tw, half * 3 * F::WORDS * 4, si))) return rc;
    c.begin(PK_OTHER, si, TAU_TABLE_ELEMS);
    k_fft_stage_root<Fr><<<1, 32, 0, st>>>(d_root, two_adicity - (log_ns + 1), d_stage);
    k_tau_tables<Fr><<<div_up(TAU_TABLE_ELEMS, 128), 128, 0, st>>>(d_stage, d_stage + Fr::L, 0, d_table);
    c.end(si);
    VecBatch b;
    memset(&b, 0, sizeof b);
    b.seg[0].in = d_x + half * C::SIZE_U; b.seg[0].n = (uint32_t)half; b.nseg = 1; b.total = (uint32_t)half;
    const uint32_t mask = (1u << log_ns) - 1, shift = (uint32_t)__builtin_ctzll(row_len);
    c.begin(G::GROUP == 0 ? PK_BATCH_EXP_G1 : PK_BATCH_EXP_G2, si, half);
    using GC = typename CoopOf<G>::type;
    bool coop = false;
    if constexpr (!std::is_void<GC>::value) {
      if (coop_g2_enabled<GC>()) {
        coop = true;
        if (ExpBlock<GC>::SMEM > 48 * 1024)
          CUDA_TRY(cudaFuncSetAttribute(k_fft_row_twiddle<GC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ExpBlock<GC>::SMEM));
        k_fft_row_twiddle<GC><<<div_up(half, ExpBlock<GC>::PPB), EXP_BLOCK, ExpBlock<GC>::SMEM, st>>>(b, d_table, mask, shift, d_tw, d_status);
      }
    }
    if (!coop) {
      constexpr size_t TREE_BYTES = 16 + 2 * EXP_BLOCK * sizeof(typename F::T);
      if (TREE_BYTES > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(k_fft_row_twiddle<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TREE_BYTES));
      k_fft_row_twiddle<G><<<div_up(half, EXP_BLOCK), EXP_BLOCK, TREE_BYTES, st>>>(b, d_table, mask, shift, d_tw, d_status);
    }
    c.end(si);
  }
  c.begin(PK_OTHER, si, n);
  k_fft_row_butterfly<G><<<div_up(half, 128), 128, 0, st>>>((uint32_t)half, (uint32_t)row_len, log_ns, d_x, d_tw, d_jac);
  c.end(si);
  run_normalize_other<G>(c, si, d_jac, n, d_out, 0);
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

template <class G>
inline int run_points_sub(Ctx& c, int si, const uint8_t* d_hi, const uint8_t* d_lo, uint64_t n, uint8_t* d_out, uint32_t out_compressed,
                          char* err, size_t errcap) {
  if (n == 0) return SSO_OK;
  if (n > (1ull << 30)) { set_err(err, errcap, "vector too long"); return SSO_E_ARG; }
  uint32_t* d_jac;
  int rc;
  if ((rc = c.alloc((void**)&d_jac, n * 3 * G::F::WORDS * 4, si))) return rc;
  c.begin(PK_OTHER, si, n);
  k_points_sub<G><<<div_up(n, 128), 128, 0, c.s[si]>>>((uint32_t)n, d_hi, d_lo, d_jac);
  c.end(si);
  run_normalize_other<G>(c, si, d_jac, n, d_out, out_compressed);
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

template <class G1, class G2, class PP> struct CurveImpl {
  static int same_ratio(Ctx& c, int si, const uint8_t* d_checks, uint64_t n, uint32_t* d_verdicts, char* err, size_t errcap) {
    return run_same_ratio<G1, G2, PP>(c, si, d_checks, n, d_verdicts, err, errcap);
  }
  static int tau_tables(Ctx& c, int si, uint64_t first_index, const uint8_t* tau, const uint8_t* const coeffs[TAU_COEFF_SLOTS],
                        uint32_t** d_table, char* err, size_t errcap) {
    return run_tau_tables<typename G1::Fr>(c, si, first_index, tau, coeffs, d_table, err, errcap);
  }
  static int batch_exp(Ctx& c, int si, uint32_t group, const VecBatch& batch, uint32_t in_compressed, const uint32_t* d_table,
                       uint32_t out_compressed, uint32_t check, uint32_t* d_status, char* err, size_t errcap) {
    if (group == GROUP_G1) return run_batch_exp<G1>(c, si, batch, in_compressed, d_table, out_compressed, check, d_status, err, errcap);
    if (group == GROUP_G2) return run_batch_exp<G2>(c, si, batch, in_compressed, d_table, out_compressed, check, d_status, err, errcap);
    set_err(err, errcap, "unknown group %u", group);
    return SSO_E_ARG;
  }
  static int batch_exp_chunk(Ctx& c, int si, const VecBatch& b1, const VecBatch& b2, uint32_t in_compressed, const uint32_t* d_table,
                             uint32_t out_compressed, uint32_t check, uint32_t* d_status, char* err, size_t errcap) {
    return run_batch_exp_chunk<G1, G2>(c, si, b1, b2, in_compressed, d_table, out_compressed, check, d_status, err, errcap);
  }
  static int reencode(Ctx& c, int si, uint32_t group, const uint8_t* d_in, uint32_t in_compressed, uint64_t n, uint8_t* d_out,
                      uint32_t out_compressed, uint32_t check, uint32_t subgroup, uint32_t* d_aff, uint32_t* d_status, char* err,
                      size_t errcap) {
    if (group == GROUP_G1) return run_reencode<G1>(c, si, d_in, in_compressed, n, d_out, out_compressed, check, subgroup, d_aff, d_status, err, errcap);
    if (group == GROUP_G2) return run_reencode<G2>(c, si, d_in, in_compressed, n, d_out, out_compressed, check, subgroup, d_aff, d_status, err, errcap);
    set_err(err, errcap, "unknown group %u", group);
    return SSO_E_ARG;
  }
  static int msm_pairs(Ctx& c, int si, uint32_t group, const uint32_t* d_aff_a, const uint32_t* d_aff_b, uint64_t n,
                       const uint8_t seed32[32], const uint64_t* tweak, uint8_t* d_out, char* err, size_t errcap) {
    if (group == GROUP_G1) return run_msm_pairs<G1>(c, si, d_aff_a, d_aff_b, n, seed32, tweak, d_out, err, errcap);
    if (group == GROUP_G2) return run_msm_pairs<G2>(c, si, d_aff_a, d_aff_b, n, seed32, tweak, d_out, err, errcap);
    set_err(err, errcap, "unknown group %u", group);
    return SSO_E_ARG;
  }
  static int keygen_g1(Ctx& c, int si, const uint32_t* d_seed, uint32_t nscalars, uint32_t* d_scalars, uint8_t* d_g1, char* err, size_t errcap) {
    if (nscalars < 1 || nscalars > 3) { set_err(err, errcap, "keygen: 1..3 scalars"); return SSO_E_ARG; }
    c.begin(PK_OTHER, si, nscalars);
    k_keygen_g1<G1><<<1, 96, 0, c.s[si]>>>(d_seed, nscalars, d_scalars, d_g1);
    c.end(si);
    CUDA_TRY(cudaGetLastError());
    return SSO_OK;
  }
  static int keygen_scalars(Ctx& c, int si, const uint32_t* d_seed, uint32_t nscalars, uint32_t* d_scalars, char* err, size_t errcap) {
    if (nscalars < 1 || nscalars > 3) { set_err(err, errcap, "keygen: 1..3 scalars"); return SSO_E_ARG; }
    c.begin(PK_OTHER, si, nscalars);
    k_keygen_scalars<G1><<<1, 32, 0, c.s[si]>>>(d_seed, nscalars, d_scalars);
    c.end(si);
    CUDA_TRY(cudaGetLastError());
    return SSO_OK;
  }
  static int hash_to_g2(Ctx& c, int si, uint32_t n, const uint32_t* d_seeds, const uint32_t* d_scalars, uint8_t* d_g2_s, uint8_t* d_g2_sx,
                        char* err, size_t errcap) {
    if (n == 0) return SSO_OK;
    c.begin(PK_OTHER, si, n);
    k_hash_to_g2<G2><<<n, 32, 0, c.s[si]>>>(n, d_seeds, d_scalars, d_g2_s, d_g2_sx);
    c.end(si);
    CUDA_TRY(cudaGetLastError());
    return SSO_OK;
  }
  static int points_sum(Ctx& c, int si, uint32_t group, const uint8_t* d_points, uint32_t n, uint8_t* d_out, uint32_t* d_status, char* err, size_t errcap) {
    if (group == GROUP_G1) return run_points_sum<G1>(c, si, d_points, n, d_out, d_status, err, errcap);
    if (group == GROUP_G2) return run_points_sum<G2>(c, si, d_points, n, d_out, d_status, err, errcap);
    set_err(err, errcap, "unknown group %u", group);
    return SSO_E_ARG;
  }
  static int fill_generator(Ctx& c, int si, uint32_t group, uint64_t n, uint8_t* d_out, uint32_t out_compressed, char* err, size_t errcap) {
    if (group == GROUP_G1) return run_fill_generator<G1>(c, si, n, d_out, out_compressed, err, errcap);
    if (group == GROUP_G2) return run_fill_generator<G2>(c, si, n, d_out, out_compressed, err, errcap);
    set_err(err, errcap, "unknown group %u", group);
    return SSO_E_ARG;
  }
  static int group_fft(Ctx& c, int si, uint32_t group, const uint8_t* d_x, uint32_t log_n, const uint32_t* root, uint32_t two_adicity,
                       const uint8_t* scale, uint8_t* d_out, uint32_t out_compressed, uint32_t* d_status, char* err, size_t errcap) {
    if (group == GROUP_G1) return run_group_fft<G1>(c, si, d_x, log_n, root, two_adicity, scale, d_out, out_compressed, d_status, err, errcap);
    if (group == GROUP_G2) return run_group_fft<G2>(c, si, d_x, log_n, root, two_adicity, scale, d_out, out_compressed, d_status, err, errcap);
    set_err(err, errcap, "unknown group %u", group);
    return SSO_E_ARG;
  }
  static int points_sub(Ctx& c, int si, uint32_t group, const uint8_t* d_hi, const uint8_t* d_lo, uint64_t n, uint8_t* d_out,
                        uint32_t out_compressed, char* err, size_t errcap) {
    if (group == GROUP_G1) return run_points_sub<G1>(c, si, d_hi, d_lo, n, d_out, out_compressed, err, errcap);
    if (group == GROUP_G2) return run_points_sub<G2>(c, si, d_hi, d_lo, n, d_out, out_compressed, err, errcap);
    set_err(err, errcap, "unknown group %u", group);
    return SSO_E_ARG;
  }
  static int fft_part_tables(Ctx& c, int si, const uint32_t* root, uint32_t squarings, uint64_t e, const uint8_t* scale, uint32_t** d_table,
                             char* err, size_t errcap) {
    return run_fft_part_tables<typename G1::Fr>(c, si, root, squarings, e, scale, d_table, err, errcap);
  }
  static int fft_row_stage(Ctx& c, int si, uint32_t group, const uint8_t* d_x, uint64_t rows, uint64_t row_len, uint32_t log_ns, const uint32_t* root,
                           uint32_t two_adicity, uint32_t* d_status, uint8_t* d_out, char* err, size_t errcap) {
    if (group == GROUP_G1) return run_fft_row_stage<G1>(c, si, d_x, rows, row_len, log_ns, root, two_adicity, d_status, d_out, err, errcap);
    if (group == GROUP_G2) return run_fft_row_stage<G2>(c, si, d_x, rows, row_len, log_ns, root, two_adicity, d_status, d_out, err, errcap);
    set_err(err, errcap, "unknown group %u", group);
    return SSO_E_ARG;
  }
  static const CurveOps* ops() {
    static const CurveOps o = {&tau_tables, &batch_exp, &batch_exp_chunk, &reencode, &msm_pairs, &same_ratio, (uint32_t)Pairing<G1, G2, PP>::CHECK_BYTES, &keygen_g1, &keygen_scalars, &hash_to_g2, (uint32_t)G1::Fr::L, &points_sum, &fill_generator, (uint32_t)G1::Fr::NBYTES, {2u * G1::F::WORDS, 2u * G2::F::WORDS}, G2::VERIFY_WEIGHT, &group_fft, &points_sub, &fft_part_tables, &fft_row_stage};
    return &o;
  }
};

// one getter per curve, each defined in its own .cu
const CurveOps* curve_ops_bls12_377();
const CurveOps* curve_ops_bw6_761();
const CurveOps* curve_ops_mnt4_753();
const CurveOps* curve_ops_mnt6_753();

}  // namespace sso
