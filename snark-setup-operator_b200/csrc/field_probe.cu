// TEST-ONLY kernels behind sso_test_field_op (field_probe.cuh), one per field of the five curves' arithmetic.
// A translation unit of their own: instantiated beside the batch_exp kernels of a curve, they change how those kernels'
// out-of-line field functions are compiled (measured on the cooperative G2 bodies), and the product kernels must not change for
// a test hook.  tools/build_variant.sh recompiles this unit with a variant's flags, so a variant library is probed with them.
#include "host.cuh"
#include "field_probe.cuh"

namespace sso {

template <class F, class G>
__global__ void __launch_bounds__(128, 1) k_field_op(uint32_t n, const uint32_t* ops, const uint32_t* a, const uint32_t* b, const uint32_t* k,
                                                   uint32_t* out, uint32_t* rc) {
  uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
  if (tid < n) body_field_op<F, G>(tid, ops, a, b, k, out, rc);
}
// one group of DEG lanes per element, as in the batch_exp bodies: groups past n leave whole, lanes 30-31 of an Fq3 warp idle
template <class GC>
__global__ void __launch_bounds__(128, 1) k_field_op_coop(uint32_t n, const uint32_t* ops, const uint32_t* a, const uint32_t* b,
                                                        const uint32_t* k, uint32_t* out, uint32_t* rc) {
  using CO = Coop<GC::F::DEG>;
  if (!CO::lane_active()) return;
  uint32_t i = blockIdx.x * ((blockDim.x >> 5) * CO::GROUPS_PER_WARP) + CO::group_in_block();
  if (i < n) body_field_op<typename GC::F, GC>(i, ops, a, b, k, out, rc);
}

// field ids of include/sso_b200.h; d_* device arrays of n elements
int run_field_op(Ctx& c, int si, uint32_t field, const uint32_t* d_ops, const uint32_t* d_a, const uint32_t* d_b, const uint32_t* d_k,
                 uint32_t* d_out, uint32_t* d_rc, uint64_t n, char* err, size_t errcap) {
  if (n == 0) return SSO_OK;
  if (n > (1ull << 30)) { set_err(err, errcap, "too many elements"); return SSO_E_ARG; }
  const uint32_t g = div_up(n, 128), gq2 = div_up(n, 4 * Coop<2>::GROUPS_PER_WARP), gq3 = div_up(n, 4 * Coop<3>::GROUPS_PER_WARP);
  cudaStream_t st = c.s[si];
  const uint32_t m = (uint32_t)n;
  c.begin(PK_OTHER, si, n);
  switch (field) {
    case 0: k_field_op<Fr253, void><<<g, 128, 0, st>>>(m, d_ops, d_a, d_b, d_k, d_out, d_rc); break;
    case 1: k_field_op<Fq377, Bls12_377_G1><<<g, 128, 0, st>>>(m, d_ops, d_a, d_b, d_k, d_out, d_rc); break;
    case 2: k_field_op<Fq761, Bw6_761_G1><<<g, 128, 0, st>>>(m, d_ops, d_a, d_b, d_k, d_out, d_rc); break;
    case 3: k_field_op<Fq4, Mnt4_753_G1><<<g, 128, 0, st>>>(m, d_ops, d_a, d_b, d_k, d_out, d_rc); break;
    case 4: k_field_op<Fq6, Mnt6_753_G1><<<g, 128, 0, st>>>(m, d_ops, d_a, d_b, d_k, d_out, d_rc); break;
    case 5: k_field_op<Fq377x2, Bls12_377_G2><<<g, 128, 0, st>>>(m, d_ops, d_a, d_b, d_k, d_out, d_rc); break;
    case 6: k_field_op<Fq4x2, Mnt4_753_G2><<<g, 128, 0, st>>>(m, d_ops, d_a, d_b, d_k, d_out, d_rc); break;
    case 7: k_field_op<Fq6x3, Mnt6_753_G2><<<g, 128, 0, st>>>(m, d_ops, d_a, d_b, d_k, d_out, d_rc); break;
    case 8: k_field_op_coop<Bls12_377_G2C><<<gq2, 128, 0, st>>>(m, d_ops, d_a, d_b, d_k, d_out, d_rc); break;
    case 9: k_field_op_coop<Mnt4_753_G2C><<<gq2, 128, 0, st>>>(m, d_ops, d_a, d_b, d_k, d_out, d_rc); break;
    case 10: k_field_op_coop<Mnt6_753_G2C><<<gq3, 128, 0, st>>>(m, d_ops, d_a, d_b, d_k, d_out, d_rc); break;
    default: set_err(err, errcap, "unknown field %u", field); return SSO_E_ARG;
  }
  c.end(si);
  CUDA_TRY(cudaGetLastError());
  return SSO_OK;
}

}  // namespace sso
