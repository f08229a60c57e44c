// TEST-ONLY: runs the per-thread bodies of the CUDA kernels (snark-setup-operator_b200/csrc/*.cuh)
// on the CPU under an instruction-level emulation of the PTX carry flag, so that the device
// algorithms can be checked against the oracle in a container without a GPU.  This library is
// built by tests/test_emul_*.py only; the product library (libsso_b200.so) never contains it
// and has no CPU path.
#define SSO_HOST_EMUL 1
#define __device__
#define __host__
#define __global__
#define __constant__ static const
#define __forceinline__ inline
#define __noinline__ __attribute__((noinline))
#include <cstdint>
#include <cstddef>
#include <cstring>
#include <vector>
#include <algorithm>
#include <numeric>
#include "../../snark-setup-operator_b200/csrc/kernels.cuh"
#include "../../snark-setup-operator_b200/csrc/msm.cuh"
#include "../../snark-setup-operator_b200/csrc/pairing.cuh"
#include "../../snark-setup-operator_b200/csrc/keygen.cuh"
#include "../../snark-setup-operator_b200/csrc/field_probe.cuh"

using namespace sso;

template <class F> static int field_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out) {
  typename F::T x, y, r;
  uint32_t fl;
  if (!F::from_bytes(a, false, fl, x)) return -1;
  if (!F::from_bytes(b, false, fl, y)) return -1;
  int rc = 0;
  switch (op) {
    case 0: r = F::mul(x, y); break;
    case 1: r = F::add(x, y); break;
    case 2: r = F::sub(x, y); break;
    case 3: r = F::sqr(x); break;
    case 4: r = F::neg(x); break;
    case 5: r = F::inv(x); break;
    case 6: if constexpr (F::DEG == 1) r = F::sqr_dedicated(x); else r = F::sqr(x); break;
    case 7: r = x; rc = F::lex_is_neg(x) ? 1 : 0; break;
    default: return -2;
  }
  F::to_bytes(out, r, 0);
  return rc;
}

// the same operations on a cooperative extension field (coop.cuh): lane r parses, computes and writes coefficient r
template <class F> static int field_op_coop(int op, const uint8_t* a, const uint8_t* b, uint8_t* out) {
  using B = typename F::B;
  int rcs[3] = {0, 0, 0};
  coop_emu_run(F::DEG, [&](int role) {
    typename F::T x, y, r;
    uint32_t fl;
    if (!F::from_bytes(a, false, fl, x) || !F::from_bytes(b, false, fl, y)) { rcs[role] = -1; return; }
    switch (op) {
      case 0: r = F::mul(x, y); break;
      case 1: r = F::add(x, y); break;
      case 2: r = F::sub(x, y); break;
      case 3: case 6: r = F::sqr(x); break;
      case 4: r = F::neg(x); break;
      case 5: r = F::inv(x); break;
      default: rcs[role] = -2; return;
    }
    B::to_bytes(out + (size_t)role * B::NBYTES, r, 0);
  });
  return rcs[0];
}

extern "C" int emul_field_op(int field, int op, const uint8_t* a, const uint8_t* b, uint8_t* out) {
  switch (field) {
    case 8: return field_op_coop<Bls12_377_G2C::F>(op, a, b, out);
    case 9: return field_op_coop<Mnt4_753_G2C::F>(op, a, b, out);
    case 10: return field_op_coop<Mnt6_753_G2C::F>(op, a, b, out);
    case 0: return field_op<Fr253>(op, a, b, out);
    case 1: return field_op<Fq377>(op, a, b, out);
    case 2: return field_op<Fq761>(op, a, b, out);
    case 3: return field_op<Fq4>(op, a, b, out);
    case 4: return field_op<Fq6>(op, a, b, out);
    case 5: return field_op<Fq377x2>(op, a, b, out);
    case 6: return field_op<Fq4x2>(op, a, b, out);
    case 7: return field_op<Fq6x3>(op, a, b, out);
  }
  return -3;
}

// Raw-limb probes of the unreduced-operand machinery (fp.cuh "lazy operands"): operands are little-endian words that need not be
// below p.  op 0: out = mont_mul(a, b) (= a b R^-1 mod p, canonical when a b < p R); op 1: out = reduce_small(a) (a < 16 p);
// op 2: out = mad_small_lazy(a, k, b) = a + k b as integers; op 3: out = mont_sqr(a) (dedicated squaring).
template <class F> static int lazy_probe(int op, const uint32_t* a, const uint32_t* b, uint32_t k, uint32_t* out) {
  typename F::T x, y, r;
  for (int i = 0; i < F::L; i++) { x.v[i] = a[i]; y.v[i] = b[i]; }
  switch (op) {
    case 0: r = F::mul(x, y); break;
    case 1: r = F::reduce_small(x); break;
    case 2: r = F::mad_small_lazy(x, k, y); break;
    case 3: r = F::sqr_dedicated(x); break;
    default: return -2;
  }
  for (int i = 0; i < F::L; i++) out[i] = r.v[i];
  return 0;
}
extern "C" int emul_lazy_probe(int field, int op, const uint32_t* a, const uint32_t* b, uint32_t k, uint32_t* out) {
  switch (field) {
    case 1: return lazy_probe<Fq377>(op, a, b, k, out);
    case 2: return lazy_probe<Fq761>(op, a, b, k, out);
    case 3: return lazy_probe<Fq4>(op, a, b, k, out);
    case 4: return lazy_probe<Fq6>(op, a, b, k, out);
  }
  return -3;
}

// sso_test_field_op on the CPU: the same body (field_probe.cuh), the same field ids and op codes; a cooperative field runs all
// its elements on DEG lockstep lane threads
template <class F, class G> static void field_op_raw(const uint32_t* ops, const uint32_t* a, const uint32_t* b, const uint32_t* k,
                                                     uint32_t* out, uint32_t* rc, uint64_t n) {
  if constexpr (F::COOP == 0) {
    for (uint64_t i = 0; i < n; i++) body_field_op<F, G>((uint32_t)i, ops, a, b, k, out, rc);
  } else {
    coop_emu_run(F::DEG, [&](int) { for (uint64_t i = 0; i < n; i++) body_field_op<F, G>((uint32_t)i, ops, a, b, k, out, rc); });
  }
}
extern "C" int emul_field_op_raw(uint32_t field, const uint32_t* ops, const uint32_t* a, const uint32_t* b, const uint32_t* k,
                                 uint32_t* out, uint32_t* rc, uint64_t n) {
  switch (field) {
    case 0: field_op_raw<Fr253, void>(ops, a, b, k, out, rc, n); return 0;
    case 1: field_op_raw<Fq377, Bls12_377_G1>(ops, a, b, k, out, rc, n); return 0;
    case 2: field_op_raw<Fq761, Bw6_761_G1>(ops, a, b, k, out, rc, n); return 0;
    case 3: field_op_raw<Fq4, Mnt4_753_G1>(ops, a, b, k, out, rc, n); return 0;
    case 4: field_op_raw<Fq6, Mnt6_753_G1>(ops, a, b, k, out, rc, n); return 0;
    case 5: field_op_raw<Fq377x2, Bls12_377_G2>(ops, a, b, k, out, rc, n); return 0;
    case 6: field_op_raw<Fq4x2, Mnt4_753_G2>(ops, a, b, k, out, rc, n); return 0;
    case 7: field_op_raw<Fq6x3, Mnt6_753_G2>(ops, a, b, k, out, rc, n); return 0;
    case 8: field_op_raw<Bls12_377_G2C::F, Bls12_377_G2C>(ops, a, b, k, out, rc, n); return 0;
    case 9: field_op_raw<Mnt4_753_G2C::F, Mnt4_753_G2C>(ops, a, b, k, out, rc, n); return 0;
    case 10: field_op_raw<Mnt6_753_G2C::F, Mnt6_753_G2C>(ops, a, b, k, out, rc, n); return 0;
  }
  return -3;
}

// out = some sqrt of a (rc 1) or rc 0 if non-square; field ids as above but via the group configs
template <class G> static int group_sqrt(const uint8_t* a, uint8_t* out) {
  using F = typename G::F;
  typename F::T x, r;
  uint32_t fl;
  if (!F::from_bytes(a, false, fl, x)) return -1;
  if (!G::field_sqrt(x, r)) return 0;
  F::to_bytes(out, r, 0);
  return 1;
}
extern "C" int emul_group_sqrt(uint32_t curve, uint32_t group, const uint8_t* a, uint8_t* out) {
  int rc = -9;
  dispatch_group(curve, group, [&](auto g) { rc = group_sqrt<decltype(g)>(a, out); });
  return rc;
}

// G = the group configuration of the batch_exp bodies (possibly a cooperative one, coop.cuh), GN = the one-thread-per-element
// configuration of the same group for the normalisation
template <class G, class GN>
static void batch_exp_emul(const uint8_t* in, uint32_t in_compressed, uint32_t n, const uint32_t* tau_canon, const uint32_t* coeff_canon,
                           uint64_t first_index, uint32_t mode, uint32_t check, uint8_t* out, uint32_t out_compressed, uint32_t* status) {
  using Fr = typename G::Fr;
  using F = typename GN::F;
  using C = SW<GN>;
  constexpr uint32_t PPB = ExpBlock<G>::PPB;
  std::vector<uint32_t> table((size_t)TAU_TABLE_ELEMS * Fr::L);
  std::vector<uint32_t> coeffs((size_t)TAU_COEFF_SLOTS * Fr::L, 0);
  for (int i = 0; i < TAU_COEFF_SLOTS; i++) coeffs[(size_t)i * Fr::L] = 1;
  // the coefficient goes to slot 2 so that the slot plumbing is exercised too
  if (coeff_canon) memcpy(coeffs.data() + 2 * Fr::L, coeff_canon, Fr::L * 4);
  for (uint32_t t = 0; t < (uint32_t)TAU_TABLE_ELEMS; t++)
    body_tau_tables<Fr>(t, tau_canon, coeffs.data(), first_index, table.data());
  // split the vector into two segments to exercise the multi-vector launch path
  uint32_t n0 = n / 2, n1 = n - n0;
  size_t isz = in_compressed ? C::SIZE_C : C::SIZE_U, osz = out_compressed ? C::SIZE_C : C::SIZE_U;
  VecBatch b;
  memset(&b, 0, sizeof b);
  if (n0) { b.seg[b.nseg++] = VecSeg{in, out, n0, 2, coeff_canon != nullptr, mode}; }
  // second segment continues the index range: emulate by a second table start -> instead run it as its own batch
  b.total = n0;
  std::vector<uint32_t> jac((size_t)n * 3 * F::WORDS);
  for (uint32_t blk = 0; blk * PPB < n0; blk++) block_batch_exp_all<G>(blk, b, in_compressed, table.data(), check, jac.data(), status);
  for (uint32_t t = 0; t * NORM_BATCH < n0; t++) body_normalize_write<GN>(t, b, jac.data(), out_compressed);
  // remaining elements: a batch of two segments (n1 - 1 elements + 1 element) starting at index first + n0
  std::vector<uint32_t> table2((size_t)TAU_TABLE_ELEMS * Fr::L);
  for (uint32_t t = 0; t < (uint32_t)TAU_TABLE_ELEMS; t++)
    body_tau_tables<Fr>(t, tau_canon, coeffs.data(), first_index + n0, table2.data());
  uint32_t st2[3] = {0, 0, 0};
  if (n1 > 0) {
    VecBatch b2;
    memset(&b2, 0, sizeof b2);
    b2.seg[0] = VecSeg{in + n0 * isz, out + n0 * osz, n1, 2, coeff_canon != nullptr, mode};
    b2.nseg = 1; b2.total = n1;
    for (uint32_t blk = 0; blk * PPB < n1; blk++) block_batch_exp_all<G>(blk, b2, in_compressed, table2.data(), check, jac.data(), st2);
    for (uint32_t t = 0; t * NORM_BATCH < n1; t++) body_normalize_write<GN>(t, b2, jac.data(), out_compressed);
    if (status[0] == 0 && st2[0] != 0) { status[0] = st2[0]; status[1] = st2[1] + n0; }
  }
}

// group 0 / 1 = G1 / G2 (one thread per element); group 2 = G2 through the warp-cooperative bodies (uncompressed input only)
extern "C" int emul_batch_exp(uint32_t curve, uint32_t group, const uint8_t* in, uint32_t in_compressed, uint32_t n,
                              const uint32_t* tau_canon, const uint32_t* coeff_canon, uint64_t first_index, uint32_t mode,
                              uint32_t check, uint8_t* out, uint32_t out_compressed, uint32_t* status) {
  status[0] = status[1] = status[2] = 0;
  if (group == 2) {
    if (in_compressed) return -2;
    return dispatch_group(curve, 1, [&](auto g) {
      using GN = decltype(g);
      using GC = typename CoopOf<GN>::type;
      if constexpr (!std::is_void<GC>::value)
        batch_exp_emul<GC, GN>(in, 0, n, tau_canon, coeff_canon, first_index, mode, check, out, out_compressed, status);
      else status[0] = 0xdead;
    });
  }
  return dispatch_group(curve, group, [&](auto g) {
    using G = decltype(g);
    batch_exp_emul<G, G>(in, in_compressed, n, tau_canon, coeff_canon, first_index, mode, check, out, out_compressed, status);
  });
}

// Multi-vector launch: two segments with different coefficient slots / modes in one batch.
extern "C" int emul_batch_exp2(uint32_t curve, uint32_t group, const uint8_t* in0, uint32_t n0, const uint8_t* in1, uint32_t n1,
                               const uint32_t* tau_canon, const uint32_t* coeff1, const uint32_t* coeff2, uint64_t first_index,
                               uint8_t* out0, uint8_t* out1, uint32_t* status) {
  status[0] = status[1] = status[2] = 0;
  return dispatch_group(curve, group, [&](auto g) {
    using G = decltype(g);
    using Fr = typename G::Fr;
    using F = typename G::F;
    std::vector<uint32_t> table((size_t)TAU_TABLE_ELEMS * Fr::L);
    std::vector<uint32_t> coeffs((size_t)TAU_COEFF_SLOTS * Fr::L, 0);
    coeffs[0] = 1;
    memcpy(coeffs.data() + Fr::L, coeff1, Fr::L * 4);
    memcpy(coeffs.data() + 2 * Fr::L, coeff2, Fr::L * 4);
    for (uint32_t t = 0; t < (uint32_t)TAU_TABLE_ELEMS; t++) body_tau_tables<Fr>(t, tau_canon, coeffs.data(), first_index, table.data());
    VecBatch b;
    memset(&b, 0, sizeof b);
    b.seg[0] = VecSeg{in0, out0, n0, 1, 1, 0};      // tau^(first+j) * coeff1
    b.seg[1] = VecSeg{in1, out1, n1, 2, 1, 1};      // shared scalar coeff2
    b.nseg = 2; b.total = n0 + n1;
    std::vector<uint32_t> jac((size_t)b.total * 3 * F::WORDS);
    for (uint32_t blk = 0; blk * EXP_BLOCK < b.total; blk++) block_batch_exp_all<G>(blk, b, 0, table.data(), 1, jac.data(), status);
    for (uint32_t t = 0; t * NORM_BATCH < b.total; t++) body_normalize_write<G>(t, b, jac.data(), 1);
  });
}

// The G2 membership test of the 753-bit towers has two implementations — inside body_reencode (one thread per element) and in the
// cooperative kernel that follows it (body_subgroup_coop, lanes emulated by lockstep threads).  Both are run; rc = -7 if their
// reports differ.
extern "C" int emul_reencode(uint32_t curve, uint32_t group, const uint8_t* in, uint32_t in_compressed, uint32_t n,
                             uint8_t* out, uint32_t out_compressed, uint32_t check, uint32_t subgroup, uint32_t* status) {
  status[0] = status[1] = status[2] = 0;
  int mismatch = 0;
  int rc = dispatch_group(curve, group, [&](auto g) {
    using G = decltype(g);
    using F = typename G::F;
    for (uint32_t t = 0; t < n; t++)
      body_reencode<G>(t, n, in, in_compressed, out, out_compressed, check, subgroup, nullptr, status);
    using GC = typename CoopOf<G>::type;
    if constexpr (!std::is_void<GC>::value) {
      if constexpr (GC::ENDO_SUBGROUP_TEST == 4) {
        if (subgroup) {
          uint32_t st2[3] = {0, 0, 0};
          std::vector<uint32_t> aff((size_t)n * 2 * F::WORDS);
          for (uint32_t t = 0; t < n; t++)
            body_reencode<G>(t, n, in, in_compressed, nullptr, 0, check, 2, aff.data(), st2);
          uint32_t stl[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
          coop_emu_run(GC::F::DEG, [&](int r) {
            for (uint32_t t = 0; t < n; t++) body_subgroup_coop<GC>(t, n, aff.data(), nullptr, stl[r]);
          });
          if (st2[0] == 0 && stl[0][0] != 0) { st2[0] = stl[0][0]; st2[1] = stl[0][1]; }
          // the same through the uncompressed serialisation, when there is one
          uint32_t st3[3] = {st2[0], st2[1], 0};
          if (out && !out_compressed) {
            uint32_t stm[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
            coop_emu_run(GC::F::DEG, [&](int r) {
              for (uint32_t t = 0; t < n; t++) body_subgroup_coop<GC>(t, n, nullptr, out, stm[r]);
            });
            uint32_t st4[3] = {0, 0, 0};
            for (uint32_t t = 0; t < n; t++) body_reencode<G>(t, n, in, in_compressed, nullptr, 0, check, 2, nullptr, st4);
            if (st4[0] == 0 && stm[0][0] != 0) { st4[0] = stm[0][0]; st4[1] = stm[0][1]; }
            st3[0] = st4[0]; st3[1] = st4[1];
          }
          if (st2[0] != status[0] || st2[1] != status[1] || st3[0] != status[0] || st3[1] != status[1]) mismatch = 1;
        }
      }
    }
  });
  return mismatch ? -7 : rc;
}

// power_pairs on n serialized points with ChaCha20(seed) scalars; the CUB sort is replaced by std::sort.
extern "C" int emul_power_pairs(uint32_t curve, uint32_t group, const uint8_t* in, uint32_t in_compressed, uint32_t n,
                                const uint32_t* seed_words, uint32_t wb, uint8_t* out_pair, uint32_t* scalars_out, uint32_t* status) {
  status[0] = status[1] = status[2] = 0;
  return dispatch_group(curve, group, [&](auto g) {
    using G = decltype(g);
    using F = typename G::F;
    using Fr = typename G::Fr;
    constexpr int KL = RLC_WORDS;
    constexpr int SBITS = RLC_BITS;
    std::vector<uint32_t> aff((size_t)n * 2 * F::WORDS);
    for (uint32_t t = 0; t < n; t++) body_reencode<G>(t, n, in, in_compressed, nullptr, 0, 0, 0, aff.data(), status);
    uint32_t m = n - 1;
    std::vector<uint32_t> sc((size_t)m * KL);
    for (uint32_t t = 0; t < m; t++) body_random_scalars<KL, SBITS>(t, m, seed_words, sc.data());
    if (scalars_out) memcpy(scalars_out, sc.data(), sc.size() * 4);
    uint32_t nwin = (SBITS + wb - 1) / wb, nb = 1u << wb;
    uint32_t seg = nb < MSM_SEG ? nb : MSM_SEG, nseg = nb / seg;
    size_t pairs = (size_t)m * nwin;
    std::vector<uint32_t> keys(pairs), vals(pairs);
    for (uint32_t t = 0; t < m; t++) body_msm_keys<KL>(t, m, nwin, wb, sc.data(), keys.data(), vals.data());
    std::vector<size_t> order(pairs);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return keys[a] < keys[b]; });
    std::vector<uint32_t> k2(pairs), v2(pairs);
    for (size_t i = 0; i < pairs; i++) { k2[i] = keys[order[i]]; v2[i] = vals[order[i]]; }
    std::vector<uint32_t> buckets((size_t)2 * nwin * nb * 3 * F::WORDS), segs((size_t)2 * nwin * nseg * 6 * F::WORDS),
        wins((size_t)2 * nwin * 3 * F::WORDS);
    for (uint32_t t = 0; t < nwin * nb; t++)
      body_msm_buckets<G>(t, m, nwin, wb, k2.data(), v2.data(), aff.data(), aff.data() + 2 * F::WORDS, buckets.data());
    for (uint32_t t = 0; t < 2 * nwin * nseg; t++) body_msm_fold<G>(t, nwin, wb, buckets.data(), segs.data());
    for (uint32_t t = 0; t < 2 * nwin; t++) body_msm_window<G>(t, nwin, wb, segs.data(), wins.data());
    for (uint32_t t = 0; t < 2; t++) body_msm_final<G>(t, nwin, wb, wins.data(), out_pair);
  });
}

// same_ratio: verdicts[i] = 1 if e(a, d) == e(b, c), 0 if not, 0x100 + status on undecodable input
template <class G1, class G2, class PP> static void same_ratio_emul(const uint8_t* checks, uint32_t n, uint32_t* verdicts) {
  using PR = Pairing<G1, G2, PP>;
  using Fq = typename G1::F;
  for (uint32_t i = 0; i < n; i++) {
    typename PR::Ws w0, w1;
    uint32_t s0 = PR::run_side(0, w0, checks + (size_t)i * PR::CHECK_BYTES, 0);
    uint32_t s1 = PR::run_side(0, w1, checks + (size_t)i * PR::CHECK_BYTES, 1);
    if (s0 || s1) { verdicts[i] = 0x100 + (s0 ? s0 : s1); continue; }
    verdicts[i] = PR::combine_and_check(0, w0, w1) ? 1 : 0;
  }
}
extern "C" int emul_same_ratio(uint32_t curve, const uint8_t* checks, uint32_t n, uint32_t* verdicts) {
  switch (curve) {
    case 0: same_ratio_emul<Bls12_377_G1, Bls12_377_G2, PAIR_bls12_377>(checks, n, verdicts); return 0;
    case 1: same_ratio_emul<Bw6_761_G1, Bw6_761_G2, PAIR_bw6_761>(checks, n, verdicts); return 0;
    case 2: same_ratio_emul<Mnt4_753_G1, Mnt4_753_G2, PAIR_mnt4_753>(checks, n, verdicts); return 0;
    case 3: same_ratio_emul<Mnt6_753_G1, Mnt6_753_G2, PAIR_mnt6_753>(checks, n, verdicts); return 0;
  }
  return -1;
}

// key generation pieces
extern "C" int emul_keygen_g1(uint32_t curve, const uint32_t* seed, uint32_t nscalars, uint32_t* scalars_out, uint8_t* g1_out) {
  return dispatch_group(curve, 0, [&](auto g) { body_keygen_g1<decltype(g)>(seed, nscalars, scalars_out, g1_out); });
}
extern "C" int emul_hash_to_g2(uint32_t curve, uint32_t n, const uint32_t* seeds, const uint32_t* scalars, uint8_t* g2_s, uint8_t* g2_sx) {
  return dispatch_group(curve, 1, [&](auto g) {
    for (uint32_t t = 0; t < n; t++) body_hash_to_g2<decltype(g)>(t, n, seeds, scalars, g2_s, g2_sx);
  });
}
