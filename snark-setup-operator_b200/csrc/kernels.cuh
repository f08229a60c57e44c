// Per-thread bodies of the hot-path kernels (the __global__ wrappers live in sso_b200.cu).
//
//   K1 tau powers      body_tau_tables / scalar_for_index   (setup_utils::generate_powers_of_tau)
//   K2 batch_exp       body_batch_exp                        (setup_utils::batch_exp, batch_mul)
//   K3 read_batch      SW::read_uncompressed / read_compressed + checks
//   K4 write_batch     body_normalize_write                  (batch normalisation + serialisation)
// Reference call sites: phase1_cli::contribute at src/bin/contribute.rs:809-824 (SURVEY.md §3 A).
//
// The bodies take an explicit thread id so that tests/emul can run the very same code under an
// instruction-level emulation of the PTX carry flag in this GPU-less container.
#pragma once
#include <type_traits>
#include "curves.cuh"

namespace sso {

enum : uint32_t { CHECK_NO = 0, CHECK_NONZERO = 1, CHECK_FULL = 2 };   // CheckForCorrectness
// status codes written by kernels (first failure wins): code in [0], element index in [1]
enum : uint32_t { ST_OK = 0, ST_NONCANONICAL = 1, ST_BAD_FLAGS = 2, ST_NOT_ON_CURVE = 3, ST_ZERO_POINT = 4,
                  ST_NOT_IN_SUBGROUP = 5 };

__device__ __forceinline__ void report(uint32_t* status, uint32_t code, uint32_t index, uint32_t vec = 0) {
#ifdef SSO_HOST_EMUL
  if (status[0] == 0) { status[0] = code; status[1] = index; status[2] = vec; }
#else
  if (atomicCAS(&status[0], 0u, code) == 0u) { status[1] = index; status[2] = vec; }
#endif
}

// ---------------------------------------------------------------------------------------------
// K1: powers of tau.  Table layout (Montgomery Fr elements, Fr::L words each):
//   [0..256)    tau^k            [256..512)  tau^(256 k)       [512..768)  tau^(65536 k)
//   [768]       tau^first_index  [769..772)  coefficient slots (e.g. 1, alpha, beta)
// so tau^(first+j) * coeff = T[768] * T[j & 255] * T[256 + ((j >> 8) & 255)] * T[512 + (j >> 16)] * T[769 + slot]
// for j < 2^24: a two/three-level parallel prefix instead of one `pow` per index.
// ---------------------------------------------------------------------------------------------
static constexpr int TAU_COEFF_SLOTS = 3;
static constexpr int TAU_TABLE_ELEMS = 769 + TAU_COEFF_SLOTS;

// One launch covers up to four vectors of the same group ("segments"), e.g. tauG1 | alphaG1 | betaG1.
struct VecSeg {
  const uint8_t* in;      // serialized input points
  uint8_t* out;           // serialized output points
  uint32_t n;
  uint32_t coeff_slot;    // which table coefficient multiplies the scalar (mode 0) or IS the scalar (mode 1)
  uint32_t has_coeff;     // mode 0 only: 0 = plain tau powers
  uint32_t mode;          // 0 = tau^(first + j) [* coeff], 1 = one shared scalar
};
struct VecBatch {
  VecSeg seg[4];
  uint32_t nseg;
  uint32_t total;
};
// flat index -> (segment, index inside the segment)
__device__ __forceinline__ bool locate(const VecBatch& b, uint32_t tid, uint32_t& si, uint32_t& j) {
  if (tid >= b.total) return false;
  si = 0; j = tid;
#pragma unroll
  for (int s = 0; s < 3; s++) {
    if (si == (uint32_t)s && (uint32_t)s + 1 < b.nseg && j >= b.seg[s].n) { j -= b.seg[s].n; si = s + 1; }
  }
  return true;
}

template <class Fr>
__device__ __forceinline__ typename Fr::T fr_pow_u64(const typename Fr::T& a, uint64_t e) {
  typename Fr::T r = Fr::one();
  for (int i = 63; i >= 0; i--) {
    r = Fr::sqr(r);
    if ((e >> i) & 1) r = Fr::mul(r, a);
  }
  return r;
}

// tid in [0, TAU_TABLE_ELEMS): builds one table entry.  tau_canon: canonical little-endian words;
// coeff_canon: TAU_COEFF_SLOTS canonical scalars back to back.
template <class Fr>
__device__ __forceinline__ void body_tau_tables(uint32_t tid, const uint32_t* tau_canon, const uint32_t* coeff_canon,
                                                uint64_t first_index, uint32_t* table) {
  typename Fr::T tau = Fr::to_mont(Fr::from_const(tau_canon));
  typename Fr::T out;
  if (tid < 768) {
    uint32_t lvl = tid >> 8, k = tid & 255;
    out = fr_pow_u64<Fr>(tau, (uint64_t)k << (8 * lvl));
  } else if (tid == 768) {
    out = fr_pow_u64<Fr>(tau, first_index);
  } else {
    out = Fr::to_mont(Fr::from_const(coeff_canon + (size_t)(tid - 769) * Fr::L));
  }
  Fr::store(table + (size_t)tid * Fr::L, 1, out);
}

// canonical scalar for element j of the vector (words in k[0..Fr::L))
template <class Fr>
__device__ __forceinline__ void scalar_for_index(const uint32_t* table, uint32_t j, uint32_t n, bool has_coeff, uint32_t slot,
                                                 uint32_t* k) {
  typename Fr::T s = Fr::mul(Fr::load(table + 768 * Fr::L, 1), Fr::load(table + (size_t)(j & 255) * Fr::L, 1));
  if (n > 256) s = Fr::mul(s, Fr::load(table + (size_t)(256 + ((j >> 8) & 255)) * Fr::L, 1));
  if (n > 65536) s = Fr::mul(s, Fr::load(table + (size_t)(512 + ((j >> 16) & 255)) * Fr::L, 1));
  if (has_coeff) s = Fr::mul(s, Fr::load(table + (size_t)(769 + slot) * Fr::L, 1));
  s = Fr::from_mont(s);
#pragma unroll
  for (int i = 0; i < Fr::L; i++) k[i] = s.v[i];
}

// ---------------------------------------------------------------------------------------------
// One field inversion per thread block: product tree over the block's leaves in shared memory.
//   tree : 2 * BS field elements; the leaf of thread t sits at tree[BS + t] and is replaced by its inverse.
// Leaves must be non-zero.  tree_up / tree_down are the per-thread steps (also driven by tests/emul).
// ---------------------------------------------------------------------------------------------
#ifndef SSO_EXP_BLOCK
#define SSO_EXP_BLOCK 128
#endif
static constexpr int EXP_BLOCK = SSO_EXP_BLOCK;        // threads (= points) per block of the batch_exp kernels: one field inversion per block

template <class F> __device__ __forceinline__ void tree_up(typename F::T* tree, int n, int t) {
  if (t < n) tree[n + t] = F::mul(tree[2 * (n + t)], tree[2 * (n + t) + 1]);
}
template <class F> __device__ __forceinline__ void tree_down(typename F::T* tree, int n, int t) {
  if (t < n) {
    int k = n + t;
    typename F::T l = tree[2 * k], r = tree[2 * k + 1], pinv = tree[k];
    tree[2 * k] = F::mul(pinv, r);
    tree[2 * k + 1] = F::mul(pinv, l);
  }
}
#ifndef SSO_HOST_EMUL
template <class F> __device__ __forceinline__ void block_batch_inverse(typename F::T* tree, int t) {
  for (int n = EXP_BLOCK / 2; n >= 1; n >>= 1) { __syncthreads(); tree_up<F>(tree, n, t); }
  __syncthreads();
  if (t == 0) tree[1] = F::inv(tree[1]);
  for (int n = 1; n < EXP_BLOCK; n <<= 1) { __syncthreads(); tree_down<F>(tree, n, t); }
  __syncthreads();
}
#else
template <class F> inline void block_batch_inverse_all(typename F::T* tree) {
  for (int n = EXP_BLOCK / 2; n >= 1; n >>= 1) for (int t = 0; t < n; t++) tree_up<F>(tree, n, t);
  tree[1] = F::inv(tree[1]);
  for (int n = 1; n < EXP_BLOCK; n <<= 1) for (int t = 0; t < n; t++) tree_down<F>(tree, n, t);
}
#endif

// ---------------------------------------------------------------------------------------------
// K3 + K2: read one point, validate, multiply by its scalar, leave the Jacobian result in HBM.
//   jac_out : total * 3 * F::WORDS words, SoA [X|Y|Z][limb][flat point index]
//   status  : [0] first failure code, [1] element index inside its vector, [2] vector (segment) index
// Three stages around the per-block inversion (ec.cuh "staged scalar multiplication"):
//   exp_stage_a  per thread : decode + checks, scalar from the tau tables, recoding, Jacobian window table
//   (block)                  : block_batch_inverse over the threads' Z products
//   exp_stage_c  per thread : affine table, window loop with mixed additions, store
// ---------------------------------------------------------------------------------------------
template <class G> struct ExpTypes {
  using C = SW<G>;
  using Fr = typename G::Fr;
  static constexpr bool GLS4 = G::HAS_GLS4;            // 4-way psi decomposition (takes precedence over 2-way GLV)
  static constexpr bool GLS2 = G::HAS_GLS2;            // 2-way psi decomposition (MNT G2)
  static constexpr bool GLV = G::HAS_GLV && !GLS4;
  static constexpr int KBITS = [] { if constexpr (G::HAS_GLS4) return 64; else if constexpr (G::HAS_GLS2) return (int)G::Endo::GLS_KBITS; else if constexpr (G::HAS_GLV) return (int)G::Glv::KBITS; else return (int)G::Fr::P::BITS; }();
  static constexpr int KW = [] { if constexpr (G::HAS_GLS4) return 2; else if constexpr (G::HAS_GLS2) return (int)G::Endo::GLS_KW; else if constexpr (G::HAS_GLV) return (int)G::Glv::KW; else return (int)G::Fr::L; }();
  static constexpr int NW = (KBITS + 2 + 3) / 4;
  using State = std::conditional_t<GLS4, typename C::template Staged4<NW>, typename C::template Staged<GLV || GLS2, KW, NW>>;
};

// staged_src: the thread's serialized input point in shared memory (block_stage_input), or null = read it from global memory
// TWIDDLE (group FFT, body_fft_butterfly): the scalar of element j is tau^((j >> tw_shift) & tw_mask) — the table holds the powers of the
// stage's root of unity, so each butterfly gets its twiddle without a pow per point; the segment's scalar rule is not read
template <class G, bool TWIDDLE = false>
__device__ __forceinline__ typename G::F::T exp_stage_a(uint32_t tid, const VecBatch& b, uint32_t in_compressed, const uint32_t* table,
                                                        uint32_t check, uint32_t* status, typename ExpTypes<G>::State& st,
                                                        const uint8_t* staged_src = nullptr, uint32_t tw_mask = 0, uint32_t tw_shift = 0) {
  using C = SW<G>;
  using F = typename G::F;
  using Fr = typename G::Fr;
  using ET = ExpTypes<G>;
  uint32_t sidx, j;
  st.active = false;
  st.affine = false;
  if (!locate(b, tid, sidx, j)) return F::one();
  const VecSeg& sg = b.seg[sidx];
  typename C::Affine p;
  const uint8_t* src = staged_src ? staged_src : sg.in + (size_t)j * (in_compressed ? C::SIZE_C : C::SIZE_U);
  uint32_t dst;
  if constexpr (F::COOP != 0) dst = C::read_uncompressed(src, p);     // the cooperative bodies take uncompressed input only (host-selected)
  else dst = in_compressed ? C::read_compressed(src, p) : C::read_uncompressed(src, p);
  if (dst != C::DESER_OK) { report(status, dst, j, sidx); p.inf = true; }
  if (check != CHECK_NO && dst == C::DESER_OK) {
    if (p.inf) report(status, ST_ZERO_POINT, j, sidx);
    else if (check == CHECK_FULL && !in_compressed && !C::on_curve(p)) { report(status, ST_NOT_ON_CURVE, j, sidx); p.inf = true; }
  }
  uint32_t k[Fr::L];
  if constexpr (TWIDDLE) {
    scalar_for_index<Fr>(table, (j >> tw_shift) & tw_mask, tw_mask + 1, false, 0, k);
  } else if (sg.mode == 0) {
    scalar_for_index<Fr>(table, j, sg.n, sg.has_coeff != 0, sg.coeff_slot, k);
  } else {
    typename Fr::T s = Fr::from_mont(Fr::load(table + (size_t)(769 + sg.coeff_slot) * Fr::L, 1));
#pragma unroll
    for (int i = 0; i < Fr::L; i++) k[i] = s.v[i];
  }
  if constexpr (ET::GLS4) {
    uint32_t kd[4][2];
    C::template gls4_split<Fr::L>(k, kd);
#pragma unroll
    for (int d = 0; d < 4; d++) C::template bias_scalar<2, ET::NW>(kd[d], st.kb[d]);
  } else if constexpr (ET::GLS2) {
    uint32_t k0[ET::KW], k1[ET::KW];
    C::template gls2_split<Fr::L>(k, k0, k1);
    st.neg1 = false;
    st.neg2 = G::Endo::TM1_NEG;                          // psi(P) = [t - 1]P = -[mu]P when the trace is negative (MNT4-753)
    C::template bias_scalar<ET::KW, ET::NW>(k0, st.kb1);
    C::template bias_scalar<ET::KW, ET::NW>(k1, st.kb2);
  } else if constexpr (ET::GLV) {
    uint32_t k1[ET::KW], k2[ET::KW];
    C::template glv_split<typename G::Glv, Fr::L>(k, k1, k2, st.neg1, st.neg2);
    C::template bias_scalar<ET::KW, ET::NW>(k1, st.kb1);
    C::template bias_scalar<ET::KW, ET::NW>(k2, st.kb2);
  } else {
    st.neg1 = st.neg2 = false;
    C::template bias_scalar<Fr::L, ET::NW>(k, st.kb1);
  }
  return C::staged_table(st, p);
}

template <class G>
__device__ __forceinline__ void exp_stage_c(uint32_t tid, const VecBatch& b, typename ExpTypes<G>::State& st,
                                            const typename G::F::T& zinv, uint32_t* jac_out) {
  using C = SW<G>;
  using F = typename G::F;
  if (tid >= b.total) return;
  C::staged_normalise(st, zinv);
  typename C::Jac r;
  if constexpr (ExpTypes<G>::GLS4) r = C::staged_loop4(st);
  else {
    const uint32_t* beta = nullptr;
    if constexpr (ExpTypes<G>::GLV) beta = G::Glv::beta();
    r = C::staged_loop(st, beta);
  }
  // SoA: word w of coordinate c of point i sits at jac_out[(c * WORDS + w) * total + i] — a warp's stores of one word are one
  // contiguous 128-byte line (the AoS records of round 1 made every store a separate sector)
  const size_t total = b.total;
  uint32_t* o = jac_out + tid;
  F::store(o, total, r.X);
  F::store(o + (size_t)F::WORDS * total, total, r.Y);
  F::store(o + (size_t)2 * F::WORDS * total, total, r.Z);
}

#ifndef SSO_HOST_EMUL
// The serialized input points of a block (EXP_BLOCK consecutive points of one vector: a contiguous byte range of the file
// image) are brought into shared memory with coalesced 128-bit loads by the whole block; every thread then parses its own
// point from shared memory (point sizes of 95 / 190 / 285 bytes leave the per-thread records unaligned and 32 threads reading
// their records byte by byte from global memory touch 32 different lines per instruction).  The buffer is the inversion tree's
// (used later), plus 16 bytes for the alignment offset.  Returns the thread's record, or null when the block straddles two
// vectors (at most three blocks per launch: they read global memory directly).
// PPB = points per block (EXP_BLOCK, or fewer when several lanes share a point: coop.cuh), pb = this thread's point inside the block.
template <class G, int PPB = EXP_BLOCK>
__device__ __forceinline__ const uint8_t* block_stage_input(uint32_t block, const VecBatch& b, uint32_t in_compressed, uint8_t* smem,
                                                            uint32_t pb = threadIdx.x) {
  using C = SW<G>;
  const uint32_t sz = in_compressed ? C::SIZE_C : C::SIZE_U;
  const uint32_t f0 = block * PPB;
  if (f0 >= b.total) return nullptr;
  const uint32_t f1 = f0 + PPB - 1 < b.total ? f0 + PPB - 1 : b.total - 1;
  uint32_t s0, j0, s1, j1;
  locate(b, f0, s0, j0);
  locate(b, f1, s1, j1);
  if (s0 != s1) return nullptr;                                        // uniform over the block: no divergence at the barrier below
  const uint8_t* g0 = b.seg[s0].in + (size_t)j0 * sz;
  const uint32_t nbytes = (j1 - j0 + 1) * sz;
  const uint32_t head = (uint32_t)(reinterpret_cast<uintptr_t>(g0) & 15u);
  const uint8_t* ga = g0 - head;                                       // 16-byte aligned, inside the allocation (bases are 256-byte aligned)
  const uint32_t span = head + nbytes, full = span >> 4;
  const uint4* gv = reinterpret_cast<const uint4*>(ga);
  uint4* sv = reinterpret_cast<uint4*>(smem);
  for (uint32_t k = threadIdx.x; k < full; k += EXP_BLOCK) sv[k] = gv[k];
  for (uint32_t k = (full << 4) + threadIdx.x; k < span; k += EXP_BLOCK) smem[k] = ga[k];      // tail: never past the vector
  __syncthreads();
  const uint32_t tid = f0 + pb;
  return (pb < (uint32_t)PPB && tid <= f1) ? smem + head + (tid - f0) * sz : nullptr;
}

// whole block: `tree` is shared memory for 2 * EXP_BLOCK field elements (+ 16 bytes, see block_stage_input)
// Points per block of a batch_exp body: EXP_BLOCK, or EXP_BLOCK / 32 warps x the groups of one warp for the cooperative fields
template <class G> struct ExpBlock {
  static constexpr int COOP = G::F::COOP;
  static constexpr int PPB = COOP == 0 ? EXP_BLOCK : (EXP_BLOCK / 32) * (32 / (COOP == 0 ? 1 : COOP));
  // leaves of the inversion tree: the next power of two (40 points per block with three lanes per point -> 64, padded with ones)
  static constexpr int TL = PPB <= 32 ? 32 : PPB <= 64 ? 64 : 128;
  // shared memory: the inversion tree (2 TL whole elements) and, before it, the staged input bytes (+ 16 for the alignment offset)
  static constexpr size_t TREE = G::AFFINE_TABLE ? (size_t)2 * TL * G::F::WORDS * 4 : 0;
  static constexpr size_t STAGE = (size_t)PPB * 2 * G::F::NBYTES;
  static constexpr size_t SMEM = 16 + (TREE > STAGE ? TREE : STAGE);
};

// Cooperative body (coop.cuh): DEG lanes per point.  The tree holds one array of 2 PPB coefficients per role.
template <class G, bool TWIDDLE = false>
__device__ __forceinline__ void block_batch_exp_coop(uint32_t block, const VecBatch& b, const uint32_t* table, uint32_t check,
                                                     uint32_t* jac_out, uint32_t* status, unsigned char* smem, uint32_t tw_mask = 0,
                                                     uint32_t tw_shift = 0) {
  using F = typename G::F;
  using CO = Coop<F::DEG>;
  constexpr int PPB = ExpBlock<G>::PPB, TL = ExpBlock<G>::TL;
  typename ExpTypes<G>::State st;
  const bool lane_ok = CO::lane_active();
  const uint32_t pb = lane_ok ? CO::group_in_block() : 0xffffffffu;
  const uint32_t tid = lane_ok ? block * PPB + pb : 0xffffffffu;       // idle lanes locate nothing and never exchange
  const uint8_t* staged = block_stage_input<G, PPB>(block, b, 0, smem, pb);
  typename F::T leaf = exp_stage_a<G, TWIDDLE>(tid, b, 0, table, check, status, st, staged, tw_mask, tw_shift);
  __syncthreads();
  if constexpr (G::AFFINE_TABLE) {
    typename F::T* tree = reinterpret_cast<typename F::T*>(smem) + (size_t)(lane_ok ? CO::role() : 0) * 2 * TL;
    if (lane_ok) {
      tree[TL + pb] = leaf;
      if (PPB < TL && pb + PPB < (uint32_t)TL) tree[TL + PPB + pb] = F::one();      // padding leaves (TL - PPB <= PPB)
    }
    static_assert(TL - PPB <= PPB, "one padding leaf per group at most");
    for (int n = TL / 2; n >= 1; n >>= 1) { __syncthreads(); if (lane_ok) tree_up<F>(tree, n, (int)pb); }
    __syncthreads();
    if (lane_ok && pb == 0) tree[1] = F::inv(tree[1]);
    for (int n = 1; n < TL; n <<= 1) { __syncthreads(); if (lane_ok) tree_down<F>(tree, n, (int)pb); }
    __syncthreads();
    if (lane_ok) leaf = tree[TL + pb];
  }
  if (lane_ok) exp_stage_c<G>(tid, b, st, leaf, jac_out);
}

template <class G, bool TWIDDLE = false>
__device__ __forceinline__ void block_batch_exp(uint32_t block, const VecBatch& b, uint32_t in_compressed, const uint32_t* table,
                                                uint32_t check, uint32_t* jac_out, uint32_t* status, typename G::F::T* tree,
                                                uint32_t tw_mask = 0, uint32_t tw_shift = 0) {
  if constexpr (G::F::COOP != 0) {
    block_batch_exp_coop<G, TWIDDLE>(block, b, table, check, jac_out, status, reinterpret_cast<unsigned char*>(tree), tw_mask, tw_shift);
  } else {
    typename ExpTypes<G>::State st;
    uint32_t tid = block * EXP_BLOCK + threadIdx.x;
    const uint8_t* staged = block_stage_input<G>(block, b, in_compressed, reinterpret_cast<uint8_t*>(tree));
    typename G::F::T leaf = exp_stage_a<G, TWIDDLE>(tid, b, in_compressed, table, check, status, st, staged, tw_mask, tw_shift);
    __syncthreads();                                                  // the staged bytes are dead: the tree may take the buffer
    if constexpr (G::AFFINE_TABLE) {
      tree[EXP_BLOCK + threadIdx.x] = leaf;
      block_batch_inverse<typename G::F>(tree, threadIdx.x);
      leaf = tree[EXP_BLOCK + threadIdx.x];
    }
    exp_stage_c<G>(tid, b, st, leaf, jac_out);
  }
}
#else
// Points per block (see the device version above)
template <class G> struct ExpBlock {
  static constexpr int COOP = G::F::COOP;
  static constexpr int PPB = COOP == 0 ? EXP_BLOCK : (EXP_BLOCK / 32) * (32 / (COOP == 0 ? 1 : COOP));
  static constexpr int TL = PPB <= 32 ? 32 : PPB <= 64 ? 64 : 128;
};
// emulation of the cooperative body: the DEG lanes of a group are DEG lockstep host threads, the groups of a block run in turn
template <class G>
inline void block_batch_exp_coop_all(uint32_t block, const VecBatch& b, const uint32_t* table, uint32_t check, uint32_t* jac_out,
                                     uint32_t* status) {
  using F = typename G::F;
  constexpr int DEG = F::DEG, PPB = ExpBlock<G>::PPB, TL = ExpBlock<G>::TL;
  std::vector<typename ExpTypes<G>::State> st((size_t)PPB * DEG);
  std::vector<typename F::T> tree((size_t)DEG * 2 * TL);
  uint32_t st_local[DEG][3];
  for (int r = 0; r < DEG; r++) st_local[r][0] = st_local[r][1] = st_local[r][2] = 0;
  coop_emu_run(DEG, [&](int r) {
    typename F::T* tr = tree.data() + (size_t)r * 2 * TL;
    for (int p = 0; p < PPB; p++) tr[TL + p] = exp_stage_a<G>(block * PPB + p, b, 0, table, check, st_local[r], st[(size_t)p * DEG + r]);
    for (int p = PPB; p < TL; p++) tr[TL + p] = F::one();
    if constexpr (G::AFFINE_TABLE) {
      for (int n = TL / 2; n >= 1; n >>= 1) for (int t = 0; t < n; t++) tree_up<F>(tr, n, t);
      tr[1] = F::inv(tr[1]);
      for (int n = 1; n < TL; n <<= 1) for (int t = 0; t < n; t++) tree_down<F>(tr, n, t);
    }
    for (int p = 0; p < PPB; p++) exp_stage_c<G>(block * PPB + p, b, st[(size_t)p * DEG + r], tr[TL + p], jac_out);
  });
  if (status[0] == 0 && st_local[0][0] != 0) { status[0] = st_local[0][0]; status[1] = st_local[0][1]; status[2] = st_local[0][2]; }
}
// emulation: one block at a time, stages run for all of its threads in turn
template <class G>
inline void block_batch_exp_all(uint32_t block, const VecBatch& b, uint32_t in_compressed, const uint32_t* table, uint32_t check,
                                uint32_t* jac_out, uint32_t* status) {
  using F = typename G::F;
  if constexpr (F::COOP != 0) {
    block_batch_exp_coop_all<G>(block, b, table, check, jac_out, status);
  } else {
    std::vector<typename ExpTypes<G>::State> st(EXP_BLOCK);
    std::vector<typename F::T> tree(2 * EXP_BLOCK);
    for (int t = 0; t < EXP_BLOCK; t++)
      tree[EXP_BLOCK + t] = exp_stage_a<G>(block * EXP_BLOCK + t, b, in_compressed, table, check, status, st[t]);
    block_batch_inverse_all<F>(tree.data());
    for (int t = 0; t < EXP_BLOCK; t++) exp_stage_c<G>(block * EXP_BLOCK + t, b, st[t], tree[EXP_BLOCK + t], jac_out);
  }
}
#endif

// ---------------------------------------------------------------------------------------------
// K4: batch normalisation (Montgomery's trick over NB consecutive points per thread: one field
// inversion per NB points) and serialisation.  tid handles flat points [tid*NB, tid*NB + NB).
// ---------------------------------------------------------------------------------------------
static constexpr int NORM_BATCH = 8;

template <class G>
__device__ __forceinline__ void body_normalize_write(uint32_t tid, const VecBatch& b, const uint32_t* jac, uint32_t out_compressed) {
  using C = SW<G>;
  using F = typename G::F;
  using FT = typename F::T;
  const uint32_t n = b.total;
  // thread tid takes the points tid, tid + T, tid + 2T, ... (T = number of threads with work): with the SoA layout the
  // threads of a warp load consecutive words
  const uint32_t T = (n + NORM_BATCH - 1) / NORM_BATCH;
  if (tid >= T) return;
  const size_t total = n;
  auto zptr = [&](uint32_t idx) { return jac + (size_t)2 * F::WORDS * total + idx; };
  uint32_t cnt = 0;
  FT prefix[NORM_BATCH];
  FT acc = F::one();
  for (uint32_t i = 0; i < (uint32_t)NORM_BATCH; i++) {
    uint32_t idx = tid + i * T;
    if (idx >= n) break;
    cnt = i + 1;
    FT z = F::load(zptr(idx), total);
    prefix[i] = acc;
    if (!F::is_zero(z)) acc = F::mul(acc, z);
  }
  FT inv = F::inv(acc);
  for (int i = (int)cnt - 1; i >= 0; i--) {
    uint32_t idx = tid + (uint32_t)i * T;
    typename C::Jac p{F::load(jac + idx, total), F::load(jac + (size_t)F::WORDS * total + idx, total), F::load(zptr(idx), total)};
    typename C::Affine a;
    if (F::is_zero(p.Z)) {
      a.inf = true; a.x = F::zero(); a.y = F::zero();
    } else {
      FT zinv = F::mul(inv, prefix[i]);
      inv = F::mul(inv, p.Z);
      a = C::to_affine_with(p, zinv);
    }
    uint32_t sidx, j;
    locate(b, idx, sidx, j);
    uint8_t* out = b.seg[sidx].out;
    if (out_compressed) C::write_compressed(out + (size_t)j * C::SIZE_C, a);
    else C::write_uncompressed(out + (size_t)j * C::SIZE_U, a);
  }
}

// ---------------------------------------------------------------------------------------------
// Group FFT (prepare_phase2: the Lagrange-basis transform of phase-2 setup): radix-2 Stockham stages, natural order in and out.
// Stage s (Ns = 2^s) over n points x (uncompressed) takes, for each j < n / 2,
//   a = x[j],  t = w^(j mod Ns) x[j + n/2]  (w = the root of unity of order 2 Ns; t from the twiddle batch_exp: exp_stage_a
//   TWIDDLE over the upper half, Jacobian SoA, n / 2 points; stage 0 has only the trivial twiddle 1 and reads x[j + n/2] itself)
// and writes a + t to o = 2 Ns floor(j / Ns) + (j mod Ns) and a - t to o + Ns (Jacobian SoA, n points) for body_normalize_write.
// The Jacobian additions are the complete ones: a = t doubles, a = -t and infinity give the identity.
// ---------------------------------------------------------------------------------------------
template <class G>
__device__ __forceinline__ void body_fft_butterfly(uint32_t j, uint32_t half, uint32_t log_ns, const uint8_t* x, const uint32_t* tw,
                                                   uint32_t* jac_out) {
  using C = SW<G>;
  using F = typename G::F;
  if (j >= half) return;
  typename C::Affine pa, pb;
  C::read_uncompressed(x + (size_t)j * C::SIZE_U, pa);
  typename C::Jac a = C::from_affine(pa), t;
  if (tw) {
    t.X = F::load(tw + j, half);
    t.Y = F::load(tw + (size_t)F::WORDS * half + j, half);
    t.Z = F::load(tw + (size_t)2 * F::WORDS * half + j, half);
  } else {
    C::read_uncompressed(x + ((size_t)j + half) * C::SIZE_U, pb);
    t = C::from_affine(pb);
  }
  const typename C::Jac s = C::add(a, t), d = C::add(a, C::neg(t));
  const uint32_t ns = 1u << log_ns;
  const uint32_t o = ((j >> log_ns) << (log_ns + 1)) + (j & (ns - 1));
  const size_t n = (size_t)2 * half;
  uint32_t* base = jac_out + o;
  F::store(base, n, s.X);
  F::store(base + (size_t)F::WORDS * n, n, s.Y);
  F::store(base + (size_t)2 * F::WORDS * n, n, s.Z);
  base += ns;
  F::store(base, n, d.X);
  F::store(base + (size_t)F::WORDS * n, n, d.Y);
  F::store(base + (size_t)2 * F::WORDS * n, n, d.Z);
}

// The cross-part FFT of the four-step group FFT (p2prep.cuh): the stage above over rows of row_len points instead of single points.
// x holds 2 half points (uncompressed), row r at [r row_len, (r + 1) row_len).  For e < half, row j = e / row_len, column col:
//   a = x[e],  t = w^(j mod Ns) x[e + half] (tw: the twiddle batch_exp over the upper half with the row index as exponent, Jacobian SoA;
//   null in stage 0, whose twiddle is 1);  a + t to row o = 2 Ns floor(j / Ns) + (j mod Ns), a - t to row o + Ns, column col.
template <class G>
__device__ __forceinline__ void body_fft_row_butterfly(uint32_t e, uint32_t half, uint32_t row_len, uint32_t log_ns, const uint8_t* x,
                                                       const uint32_t* tw, uint32_t* jac_out) {
  using C = SW<G>;
  using F = typename G::F;
  if (e >= half) return;
  const uint32_t j = e / row_len, col = e - j * row_len;
  typename C::Affine pa, pb;
  C::read_uncompressed(x + (size_t)e * C::SIZE_U, pa);
  typename C::Jac a = C::from_affine(pa), t;
  if (tw) {
    t.X = F::load(tw + e, half);
    t.Y = F::load(tw + (size_t)F::WORDS * half + e, half);
    t.Z = F::load(tw + (size_t)2 * F::WORDS * half + e, half);
  } else {
    C::read_uncompressed(x + ((size_t)e + half) * C::SIZE_U, pb);
    t = C::from_affine(pb);
  }
  const typename C::Jac s = C::add(a, t), d = C::add(a, C::neg(t));
  const uint32_t ns = 1u << log_ns;
  const uint32_t o = ((j >> log_ns) << (log_ns + 1)) + (j & (ns - 1));
  const size_t n = (size_t)2 * half;
  uint32_t* base = jac_out + (size_t)o * row_len + col;
  F::store(base, n, s.X);
  F::store(base + (size_t)F::WORDS * n, n, s.Y);
  F::store(base + (size_t)2 * F::WORDS * n, n, s.Z);
  base += (size_t)ns * row_len;
  F::store(base, n, d.X);
  F::store(base + (size_t)F::WORDS * n, n, d.Y);
  F::store(base + (size_t)2 * F::WORDS * n, n, d.Z);
}

// h_g1 of prepare_phase2: out[j] = hi[j] - lo[j] (uncompressed inputs) as Jacobian SoA over n points
template <class G>
__device__ __forceinline__ void body_points_sub(uint32_t j, uint32_t n, const uint8_t* hi, const uint8_t* lo, uint32_t* jac_out) {
  using C = SW<G>;
  using F = typename G::F;
  if (j >= n) return;
  typename C::Affine ph, pl;
  C::read_uncompressed(hi + (size_t)j * C::SIZE_U, ph);
  C::read_uncompressed(lo + (size_t)j * C::SIZE_U, pl);
  const typename C::Jac r = C::add(C::from_affine(ph), C::neg(C::from_affine(pl)));
  F::store(jac_out + j, n, r.X);
  F::store(jac_out + (size_t)F::WORDS * n + j, n, r.Y);
  F::store(jac_out + (size_t)2 * F::WORDS * n + j, n, r.Z);
}

// ---------------------------------------------------------------------------------------------
// K3 alone: re-encode points (compressed -> uncompressed and so on) with validation — the
// decompression half of transform_pok_and_correctness / combine (SURVEY.md §8a rows a5, a8).
//   check         : CHECK_NO / CHECK_NONZERO (reject infinity) / CHECK_FULL (+ on the curve, for uncompressed input)
//   subgroup != 0 : additionally require [r]P = O (SW::in_subgroup: endomorphism form where the curve has one; nothing to do
//                   on the prime-order groups), independently of `check`
// Optionally leaves the affine Montgomery coordinates in `aff_out` ([point][x|y] words, inf -> all-zero)
// for the MSM that follows.
// ---------------------------------------------------------------------------------------------
template <class G>
__device__ __forceinline__ void body_reencode(uint32_t tid, uint32_t n, const uint8_t* in, uint32_t in_compressed,
                                              uint8_t* out, uint32_t out_compressed, uint32_t check, uint32_t subgroup,
                                              uint32_t* aff_out, uint32_t* status) {
  using C = SW<G>;
  using F = typename G::F;
  if (tid >= n) return;
  typename C::Affine p;
  uint32_t st = in_compressed ? C::read_compressed(in + (size_t)tid * C::SIZE_C, p)
                              : C::read_uncompressed(in + (size_t)tid * C::SIZE_U, p);
  if (st != C::DESER_OK) { report(status, st, tid); p.inf = true; p.x = F::zero(); p.y = F::zero(); }
  else if (p.inf) {
    if (check != CHECK_NO) report(status, ST_ZERO_POINT, tid);
  } else {
    // CheckForCorrectness and SubgroupCheckMode are independent knobs of the reference (src/bin/contribute.rs:971-984):
    // `check` decides non-zero / on-curve, `subgroup` decides the membership test.  A decompressed point is on the curve by
    // construction; an uncompressed one is checked whenever the membership test (which assumes a curve point) follows.
    // subgroup == 2: the membership test runs in the cooperative kernel that follows (body_subgroup_coop)
    if (!in_compressed && (check == CHECK_FULL || subgroup) && !C::on_curve(p)) report(status, ST_NOT_ON_CURVE, tid);
    else if (subgroup == 1 && !C::in_subgroup(p)) report(status, ST_NOT_IN_SUBGROUP, tid);
  }
  if (out) {
    if (out_compressed) C::write_compressed(out + (size_t)tid * C::SIZE_C, p);
    else C::write_uncompressed(out + (size_t)tid * C::SIZE_U, p);
  }
  if (aff_out) {
    uint32_t* o = aff_out + (size_t)tid * 2 * F::WORDS;
    F::store(o, 1, p.inf ? F::zero() : p.x);
    F::store(o + F::WORDS, 1, p.inf ? F::zero() : p.y);
  }
}

// ---------------------------------------------------------------------------------------------
// K3b: the membership test of decoded points through the warp-cooperative fields (coop.cuh): DEG lanes per point, the same
// SW::in_subgroup template.  Points come from the array the decoding kernel left: affine Montgomery words ([point][x|y], all-zero
// = infinity) when `aff` is given, else the uncompressed serialisation.  Points the decoding kernel rejected were reported
// there (first report wins); infinity is skipped.
// ---------------------------------------------------------------------------------------------
template <class GC>
__device__ __forceinline__ void body_subgroup_coop(uint32_t point, uint32_t n, const uint32_t* aff, const uint8_t* pts, uint32_t* status) {
  using C = SW<GC>;
  using F = typename GC::F;
  if (point >= n) return;
  typename C::Affine p;
  if (aff) {
    const uint32_t* a = aff + (size_t)point * 2 * F::WORDS;
    p.x = F::load(a, 1);
    p.y = F::load(a + F::WORDS, 1);
    p.inf = F::is_zero(p.x) && F::is_zero(p.y);
  } else {
    if (C::read_uncompressed(pts + (size_t)point * C::SIZE_U, p) != C::DESER_OK) return;
  }
  if (p.inf) return;
  if (!C::in_subgroup(p)) report(status, ST_NOT_IN_SUBGROUP, point);
}

}  // namespace sso
