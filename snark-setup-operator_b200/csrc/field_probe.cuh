// TEST-ONLY: one field operation per element on raw Montgomery words, the body behind sso_test_field_op (one kernel per field,
// field_probe.cu) and emul_field_op_raw (tests/emul).  Operands are loaded as they are — no to_mont, no range check — so that
// unreduced operands can be fed exactly where a contract admits them, and the result words are stored as the arithmetic
// returns them, so a test sees the representation as well as the value.
#pragma once
#include <type_traits>
#include "curves.cuh"

namespace sso {

// op codes (tests/field_cases.py keeps the table of supported (field, op) pairs)
enum : uint32_t {
  FOP_MUL = 0, FOP_ADD = 1, FOP_SUB = 2, FOP_SQR = 3, FOP_NEG = 4, FOP_INV = 5, FOP_SQR_DEDICATED = 6, FOP_LEX_IS_NEG = 7,
  FOP_SQRT = 8, FOP_REDUCE_SMALL = 9, FOP_MAD_SMALL_LAZY = 10, FOP_CONJ = 11, FOP_MUL_BASE = 12, FOP_MUL_U2 = 13, FOP_FROB_W = 14
};
// rc of an element whose (field, op) pair has no implementation: the output words are left untouched
static constexpr uint32_t FOP_RC_UNSUPPORTED = 0xffffffffu;

// Element i of one field: out = op(a, b) (k: the small factor of mad_small_lazy), rc = predicate result (lex_is_neg, sqrt found)
// or 0.  G: the group configuration whose field_sqrt is reached by FOP_SQRT, or void (a field without a group: Fp::sqrt).
// Cooperative fields (F::COOP > 0): every lane of the element's group calls this with the same i; lane r loads and stores
// coefficient r.
template <class F, class G>
__device__ __forceinline__ void body_field_op(uint32_t i, const uint32_t* ops, const uint32_t* a, const uint32_t* b, const uint32_t* k,
                                              uint32_t* out, uint32_t* rc) {
  using B = typename F::Base;
  const size_t off = (size_t)i * F::WORDS;
  const typename F::T x = F::load(a + off, 1), y = F::load(b + off, 1);
  typename F::T r = x;
  uint32_t code = 0;
  bool done = true;
  switch (ops[i]) {
    case FOP_MUL: r = F::mul(x, y); break;
    case FOP_ADD: r = F::add(x, y); break;
    case FOP_SUB: r = F::sub(x, y); break;
    case FOP_SQR: r = F::sqr(x); break;
    case FOP_NEG: r = F::neg(x); break;
    case FOP_INV: r = F::inv(x); break;
    case FOP_SQR_DEDICATED:
      if constexpr (F::DEG == 1) r = F::sqr_dedicated(x); else r = F::sqr(x);
      break;
    case FOP_LEX_IS_NEG:
      if constexpr (F::COOP == 0) code = F::lex_is_neg(x) ? 1u : 0u; else done = false;
      break;
    case FOP_SQRT:
      if constexpr (F::COOP == 0) {
        if constexpr (std::is_void<G>::value) code = F::sqrt(x, r) ? 1u : 0u;
        else code = G::field_sqrt(x, r) ? 1u : 0u;
      } else done = false;
      break;
    case FOP_REDUCE_SMALL:
      if constexpr (F::DEG == 1 && F::LAZY_OK) r = F::reduce_small(x); else done = false;
      break;
    case FOP_MAD_SMALL_LAZY:
      if constexpr (F::DEG == 1 && F::LAZY_OK) r = F::mad_small_lazy(x, k[i], y); else done = false;
      break;
    case FOP_CONJ:
      if constexpr (F::DEG == 2) r = F::conj(x); else done = false;
      break;
    case FOP_MUL_BASE:                                       // x times the base-field element held in the first coefficient of b
      if constexpr (F::DEG > 1) r = F::mul_base(x, B::load(b + off, 1)); else done = false;
      break;
    case FOP_MUL_U2:
      if constexpr (F::DEG == 3) r = F::mul_u2(x); else done = false;
      break;
    case FOP_FROB_W:
      if constexpr (F::DEG == 3 && !std::is_void<G>::value) r = F::frob_w(x, G::Endo::w1(), G::Endo::w2()); else done = false;
      break;
    default: done = false;
  }
  bool lead = true;
  if constexpr (F::COOP > 0) lead = Coop<F::COOP>::role() == 0;
  if (!done) {
    if (lead) rc[i] = FOP_RC_UNSUPPORTED;
    return;
  }
  F::store(out + off, 1, r);
  if (lead) rc[i] = code;
}

}  // namespace sso
