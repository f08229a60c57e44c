// prepare_phase2: the hand-off from phase 1 to phase 2 (phase2_cli::prepare_phase2, reached from the operator's
// intermediate_transform binary, src/bin/intermediate_transform.rs:213-226; SURVEY.md §2 row 14).  A Full-mode Groth16 powers of
// tau accumulator becomes the Lagrange-basis parameters that phase 2 is built from, by a radix-2 group FFT per vector
// (curve_ops.cuh run_group_fft; kernels.cuh body_fft_butterfly).
//
// Input : hash[64] | tauG1[2^(p+1) - 1] | tauG2[2^p] | alphaTauG1[2^p] | betaTauG1[2^p] | betaG2, uncompressed (Full mode).
// Output: for the phase-2 size m (a power of two, m <= 2^p), with IFFT(x)_i = m^-1 sum_j w^(-ij) x_j and w the generator of the
//         size-m radix-2 domain:
//           alpha_g1 = alphaTauG1[0] | beta_g1 = betaTauG1[0] | beta_g2 = betaG2
//           | coeffs_g1 = IFFT(tauG1[0..m)) (= L_i(tau) G1) | coeffs_g2 = IFFT(tauG2[0..m)) | alpha_coeffs_g1 = IFFT(alphaTauG1[0..m))
//           | beta_coeffs_g1 = IFFT(betaTauG1[0..m)) | h_g1[i] = tauG1[i + m] - tauG1[i] (i < m - 1; = tau^i (tau^m - 1) G1)
//         Every output point is determined by the input, whatever order the FFT runs in.
//
// [UP] Recalled upstream behaviour, not verifiable in the build image (tests/golden/PREPARE_PHASE2_RECIPE.md is the way to pin it):
//   - the output is the setup_utils::Groth16Params writer in the order above, uncompressed, with no length prefixes;
//   - w = GENERATOR^((r - 1) / m) with ark-ff's FftField::GENERATOR: BLS12-377 Fr 22, BW6-761 Fr 15, MNT4-753 Fr 17,
//     MNT6-753 Fr 17 (tools/gen_constants.py FR_GENERATOR; ark-poly Radix2EvaluationDomain).  A different generator permutes
//     the Lagrange basis without breaking any identity;
//   - the reference's `phase2_size` is taken as the count m (not its logarithm); anything but a power of two is rejected;
//   - the reference reads the accumulator with CheckForCorrectness::Full: every element the transform reads is checked to be
//     non-zero, on the curve and in the prime-order subgroup.
// MNT6-753 Fr has 2-adicity 15: beyond m = 2^15 arkworks switches to a mixed-radix domain, which is not implemented here.
#pragma once

namespace sso {

struct FftDomain { const uint32_t* root; const uint32_t* root_inv; const uint32_t* modulus; uint32_t two_adicity; uint32_t L; };
inline bool fft_domain(uint32_t curve, FftDomain& d) {
  switch (curve) {
    case SSO_CURVE_BLS12_377: d = {FFT_bls12_377::host_root(), FFT_bls12_377::host_root_inv(), P_r253::host_p(), FFT_bls12_377::TWO_ADICITY, P_r253::L}; return true;
    case SSO_CURVE_BW6_761: d = {FFT_bw6_761::host_root(), FFT_bw6_761::host_root_inv(), P_q377::host_p(), FFT_bw6_761::TWO_ADICITY, P_q377::L}; return true;
    case SSO_CURVE_MNT4_753: d = {FFT_mnt4_753::host_root(), FFT_mnt4_753::host_root_inv(), P_q6::host_p(), FFT_mnt4_753::TWO_ADICITY, P_q6::L}; return true;
    case SSO_CURVE_MNT6_753: d = {FFT_mnt6_753::host_root(), FFT_mnt6_753::host_root_inv(), P_q4::host_p(), FFT_mnt6_753::TWO_ADICITY, P_q4::L}; return true;
  }
  return false;
}

// canonical little-endian bytes of m^-1 mod r for m = 2^log_m dividing r - 1: m (r - 1) / m = -1, so m^-1 = r - (r - 1) / m
inline std::vector<uint8_t> fft_inv_size(const FftDomain& d, uint32_t log_m, size_t nbytes) {
  std::vector<uint32_t> q(d.modulus, d.modulus + d.L), w(d.L);
  q[0] -= 1;                                                          // r is odd
  for (uint32_t s = 0; s < log_m; s++) {
    for (uint32_t i = 0; i + 1 < d.L; i++) q[i] = (q[i] >> 1) | (q[i + 1] << 31);
    q[d.L - 1] >>= 1;
  }
  uint64_t borrow = 0;
  for (uint32_t i = 0; i < d.L; i++) {
    uint64_t t = (uint64_t)d.modulus[i] - q[i] - borrow;
    w[i] = (uint32_t)t;
    borrow = (t >> 32) & 1;
  }
  std::vector<uint8_t> out(nbytes, 0);
  memcpy(out.data(), w.data(), nbytes);
  return out;
}

inline int log2_exact(uint64_t m) {
  if (m == 0 || (m & (m - 1))) return -1;
  int l = 0;
  while ((1ull << l) < m) l++;
  return l;
}

inline size_t p2prep_size(const CurveSizes& cs, uint64_t m) { return (2 + 3 * m + (m - 1)) * cs.g1u + (1 + m) * cs.g2u; }

// the checks of prepare_phase2 that need no accumulator bytes: Full mode and Groth16, then the phase-2 size
inline int p2prep_check(const sso_p1_params_t* p, uint64_t m, P1Layout& L, FftDomain& d, int& log_m, char* err, size_t errcap) {
  int rc = p1_layout(p, L, err, errcap);
  if (rc) return rc;
  if (p->contribution_mode != SSO_MODE_FULL) { set_err(err, errcap, "prepare_phase2 reads a Full-mode accumulator (got Chunked parameters)"); return SSO_E_ARG; }
  fft_domain(p->curve, d);
  log_m = log2_exact(m);
  if (log_m < 0) { set_err(err, errcap, "phase-2 size %llu is not a power of two", (unsigned long long)m); return SSO_E_ARG; }
  if (m > L.powers_length) { set_err(err, errcap, "phase-2 size %llu exceeds the 2^%u powers of the accumulator", (unsigned long long)m, p->power); return SSO_E_ARG; }
  if ((uint32_t)log_m > d.two_adicity || log_m > 24) {
    set_err(err, errcap, "phase-2 size 2^%d is beyond the radix-2 domain of this curve's scalar field (at most 2^%u%s)", log_m,
            d.two_adicity < 24 ? d.two_adicity : 24u, d.two_adicity < 24 ? "; larger sizes need the mixed-radix domain, not supported" : "");
    return SSO_E_ARG;
  }
  return SSO_OK;
}

// The transform on a validated layout: the prefixes the transform reads are staged and checked on stream 0, then the G2 FFT runs
// on stream 1 beside the three G1 FFTs and h_g1 on stream 0.
inline int p2_prepare(Ctx& c, const CurveOps* ops, const P1Layout& L, const FftDomain& d, int log_m, const uint8_t* acc, uint8_t* out,
                      char* err, size_t errcap) {
  const CurveSizes& cs = L.cs;
  const uint64_t m = 1ull << log_m;
  int rc;
  // staged prefixes: tauG1[0 .. 2m - 1) (h_g1 reads up to index 2m - 2), tauG2 / alphaTauG1 / betaTauG1 [0 .. m), betaG2
  const uint64_t cnt[5] = {2 * m - 1, m, m, m, 1};
  static const uint32_t grp[5] = {GROUP_G1, GROUP_G2, GROUP_G1, GROUP_G1, GROUP_G2};
  uint8_t* d_in[5];
  uint32_t* d_status;
  if ((rc = status_buffer(c, &d_status, 0, false, err, errcap))) return rc;
  for (int v = 0; v < 5; v++) {
    const size_t bytes = cnt[v] * point_size(cs, grp[v], 0);
    if ((rc = c.alloc((void**)&d_in[v], bytes))) return rc;
    CUDA_TRY(cudaMemcpyAsync(d_in[v], acc + L.off_u[v], bytes, cudaMemcpyHostToDevice, c.s[0]));
    // CheckForCorrectness::Full, re-encoded in place (canonical flags for the elements copied to the output as they are)
    if ((rc = ops->reencode(c, 0, grp[v], d_in[v], 0, cnt[v], d_in[v], 0, CHECK_FULL, 1, nullptr, d_status, err, errcap))) return rc;
  }
  CUDA_TRY(cudaStreamSynchronize(c.s[0]));
  if ((rc = check_status(c, d_status, "accumulator", err, errcap))) return SSO_E_INPUT;
  // output offsets
  const size_t g1 = cs.g1u, g2 = cs.g2u;
  const size_t o_coeffs_g1 = 2 * g1 + g2, o_coeffs_g2 = o_coeffs_g1 + m * g1, o_alpha = o_coeffs_g2 + m * g2, o_beta = o_alpha + m * g1,
               o_h = o_beta + m * g1;
  std::vector<uint8_t> minv = fft_inv_size(d, (uint32_t)log_m, ops->fr_bytes);
  uint8_t *d_cg1, *d_cg2, *d_ca, *d_cb, *d_h;
  if ((rc = c.alloc((void**)&d_cg1, m * g1))) return rc;
  if ((rc = c.alloc((void**)&d_ca, m * g1))) return rc;
  if ((rc = c.alloc((void**)&d_cb, m * g1))) return rc;
  if ((rc = c.alloc((void**)&d_h, (m - 1) * g1 + 1))) return rc;
  if ((rc = c.alloc((void**)&d_cg2, m * g2, 1))) return rc;
  if ((rc = c.fork(0, 1))) return rc;
  if ((rc = ops->group_fft(c, 1, GROUP_G2, d_in[1], (uint32_t)log_m, d.root_inv, d.two_adicity, minv.data(), d_cg2, 0, d_status, err, errcap))) return rc;
  CUDA_TRY(cudaMemcpyAsync(out + o_coeffs_g2, d_cg2, m * g2, cudaMemcpyDeviceToHost, c.s[1]));
  CUDA_TRY(cudaMemcpyAsync(out, d_in[2], g1, cudaMemcpyDeviceToHost, c.s[0]));
  CUDA_TRY(cudaMemcpyAsync(out + g1, d_in[3], g1, cudaMemcpyDeviceToHost, c.s[0]));
  CUDA_TRY(cudaMemcpyAsync(out + 2 * g1, d_in[4], g2, cudaMemcpyDeviceToHost, c.s[0]));
  const uint8_t* src[3] = {d_in[0], d_in[2], d_in[3]};
  uint8_t* dst[3] = {d_cg1, d_ca, d_cb};
  const size_t off[3] = {o_coeffs_g1, o_alpha, o_beta};
  for (int v = 0; v < 3; v++) {
    if ((rc = ops->group_fft(c, 0, GROUP_G1, src[v], (uint32_t)log_m, d.root_inv, d.two_adicity, minv.data(), dst[v], 0, d_status, err, errcap))) return rc;
    CUDA_TRY(cudaMemcpyAsync(out + off[v], dst[v], m * g1, cudaMemcpyDeviceToHost, c.s[0]));
  }
  if ((rc = ops->points_sub(c, 0, GROUP_G1, d_in[0] + m * g1, d_in[0], m - 1, d_h, 0, err, errcap))) return rc;
  if (m > 1) CUDA_TRY(cudaMemcpyAsync(out + o_h, d_h, (m - 1) * g1, cudaMemcpyDeviceToHost, c.s[0]));
  if ((rc = sync_all(c, err, errcap))) return rc;
  return check_status(c, d_status, "prepare_phase2", err, errcap);
}

}  // namespace sso
