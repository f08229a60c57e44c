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
#include <algorithm>
#include <functional>

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

// the checks of prepare_phase2 that need no accumulator bytes: Full mode and Groth16, then the phase-2 size (at most 2^max_log: the
// one-device transform stops at 2^24, the transform in parts at the radix-2 domain)
inline int p2prep_check(const sso_p1_params_t* p, uint64_t m, P1Layout& L, FftDomain& d, int& log_m, char* err, size_t errcap,
                        uint32_t max_log = 24) {
  int rc = p1_layout(p, L, err, errcap);
  if (rc) return rc;
  if (p->contribution_mode != SSO_MODE_FULL) { set_err(err, errcap, "prepare_phase2 reads a Full-mode accumulator (got Chunked parameters)"); return SSO_E_ARG; }
  fft_domain(p->curve, d);
  log_m = log2_exact(m);
  if (log_m < 0) { set_err(err, errcap, "phase-2 size %llu is not a power of two", (unsigned long long)m); return SSO_E_ARG; }
  if (m > L.powers_length) { set_err(err, errcap, "phase-2 size %llu exceeds the 2^%u powers of the accumulator", (unsigned long long)m, p->power); return SSO_E_ARG; }
  if ((uint32_t)log_m > d.two_adicity || (uint32_t)log_m > max_log) {
    set_err(err, errcap, "phase-2 size 2^%d is beyond the radix-2 domain of this curve's scalar field (at most 2^%u%s)", log_m,
            d.two_adicity < max_log ? d.two_adicity : max_log, d.two_adicity < max_log ? "; larger sizes need the mixed-radix domain, not supported" : "");
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

// ---------------------------------------------------------------------------------------------
// The transform in parts (sso_group_fft_parts_buf, sso_p2_prepare_devices_buf / _file): a four-step group FFT, decimation in time,
// on host buffers.  m = P M points in P parts of M, input index j = r + P c', output index k = c + M s, w the size-m root (w^-1 and
// the scale m^-1 for the inverse transform):
//   X[c + M s] = sum_r w_P^(r s) (scale w^(r c) sum_c' w_M^(c' c) x[r + P c']),  w_M = w^P, w_P = w^M.
// Pass 1, one task per part r: the size-M group FFT of x[r::P] (run_group_fft, unscaled: its stage roots depend on the stage only),
//   then Z_r[c] = scale w^(r c) Y_r[c] (a tau-power batch_exp, tau = w^r, coefficient scale), written to the output rows r M + [0, M).
// Pass 2, one task per block of columns [c0, c0 + B): the P-point FFT over the rows r M + [c0, c0 + B) of the output, Stockham stages
//   over rows (fft_row_stage: one twiddle launch per stage, the row index as exponent of the stage root), written back in place.
// The output is the exchange buffer: one barrier between the passes, no collective, no second copy.  Device memory per task is O(M).
// Twiddle multiplications per vector: (m/2)(log2 m - 2) + m, against m + (m/2)(log2 m - 1) for the transform in one piece.
// Every output point is determined by the input, so the output does not depend on P.
// ---------------------------------------------------------------------------------------------
struct PartsPlan {
  uint64_t m, P, M, B;            // points, parts, points per part, columns per block of pass 2
  uint32_t log_m, log_p;
  const uint32_t* root;           // host, canonical words: of order 2^two_adicity (its inverse for the inverse transform)
  uint32_t two_adicity;
  const uint8_t* scale;           // host, canonical Fr bytes multiplying every output (m^-1 of the inverse transform), or null
};
inline PartsPlan parts_plan(uint32_t log_m, uint32_t log_p, const uint32_t* root, uint32_t two_adicity, const uint8_t* scale) {
  PartsPlan pl;
  pl.log_m = log_m; pl.log_p = log_p;
  pl.m = 1ull << log_m; pl.P = 1ull << log_p; pl.M = pl.m >> log_p;
  // columns per block: a block holds P B <= max(M, 2^18) points (a part, or enough points to fill the device for small parts)
  pl.B = std::min(pl.M, std::max<uint64_t>(1, std::max<uint64_t>(pl.M, 1ull << 18) >> log_p));
  pl.root = root; pl.two_adicity = two_adicity; pl.scale = scale;
  return pl;
}
// one vector of a transform in parts: m uncompressed points in (host) -> out (host); vec is the index failures report
struct PartsVec { uint32_t group; const uint8_t* in; uint8_t* out; uint32_t vec; };

// Bytes of device memory of one task for a part of M points of sz bytes: the staged part and the transformed part, the FFT's two
// buffers and Jacobian scratch (~1.5 sz per point, half of it for the twiddles); a block of pass 2 holds at most max(M, 2^18) points
// and needs less per point
inline uint64_t parts_footprint(uint64_t M, size_t sz) { return 7 * std::max<uint64_t>(M, 1ull << 18) * sz + (64ull << 20); }

// The number of parts of prepare_phase2 in parts: the smallest power of two P <= m such that P >= the number of workers,
// m / P <= 2^24 and a part of the widest vector (sz bytes a point) fits the free memory of its device (cudaMemGetInfo at call
// start) divided among the workers there.
inline int choose_parts(uint32_t log_m, size_t sz, const Participants& Pt, uint32_t& log_p, char* err, size_t errcap) {
  uint64_t per_worker = ~0ull;
  int prev = 0;
  CUDA_TRY(cudaGetDevice(&prev));
  for (int dev : Pt.devices) {
    const uint64_t on_dev = (uint64_t)std::count(Pt.devices.begin(), Pt.devices.end(), dev);
    size_t avail = 0, total = 0;
    CUDA_TRY(cudaSetDevice(dev));
    CUDA_TRY(cudaMemGetInfo(&avail, &total));
    per_worker = std::min<uint64_t>(per_worker, avail / on_dev);
  }
  CUDA_TRY(cudaSetDevice(prev));
  const uint64_t workers = Pt.devices.size();
  auto fits = [&](uint32_t lp) { return log_m - lp <= 24 && parts_footprint(1ull << (log_m - lp), sz) <= per_worker; };
  log_p = 0;
  while (log_p < log_m && ((1ull << log_p) < workers || !fits(log_p))) log_p++;
  if (!fits(log_p)) {
    set_err(err, errcap, "a part of 2^%u points needs %llu bytes of device memory, %llu are free per worker", log_m - log_p,
            (unsigned long long)parts_footprint(1ull << (log_m - log_p), sz), (unsigned long long)per_worker);
    return SSO_E_CUDA;
  }
  return SSO_OK;
}

// the status of a task: a failed check of element idx of the staged run stands for element first + stride idx of vector vec
inline int parts_status(uint32_t* d_status, const char* what, uint32_t vec, uint64_t first, uint64_t stride, char* err, size_t errcap) {
  uint32_t h[4] = {0, 0, 0, 0};
  CUDA_TRY(cudaMemcpy(h, d_status, STATUS_BYTES, cudaMemcpyDeviceToHost));
  if (h[0] == 0) return SSO_OK;
  set_err(err, errcap, "%s: %s (vector %u, element %llu)", what, status_text(h[0]), vec, (unsigned long long)(first + stride * h[1]));
  return SSO_E_INPUT;
}

// n points of sz bytes at src, src + stride, ... (host) -> d_out (contiguous) on stream 0; a strided run goes through a page-locked buffer
inline int gather_h2d(Ctx& c, const uint8_t* src, size_t stride, size_t sz, uint64_t n, uint8_t* d_out, char* err, size_t errcap) {
  if (stride == sz) {
    CUDA_TRY(cudaMemcpyAsync(d_out, src, n * sz, cudaMemcpyHostToDevice, c.s[0]));
    return SSO_OK;
  }
  const uint64_t per = std::min<uint64_t>(n, std::max<uint64_t>(1, (64ull << 20) / sz));
  PinnedLease buf(per * sz);
  if (!buf.b.p) { set_err(err, errcap, "cannot allocate %llu bytes of page-locked memory", (unsigned long long)(per * sz)); return SSO_E_CUDA; }
  for (uint64_t i0 = 0; i0 < n; i0 += per) {
    const uint64_t k = std::min(per, n - i0);
    CUDA_TRY(cudaStreamSynchronize(c.s[0]));                          // the previous run has left the buffer
    for (uint64_t i = 0; i < k; i++) memcpy(buf.b.p + i * sz, src + (i0 + i) * stride, sz);
    CUDA_TRY(cudaMemcpyAsync(d_out + i0 * sz, buf.b.p, k * sz, cudaMemcpyHostToDevice, c.s[0]));
  }
  CUDA_TRY(cudaStreamSynchronize(c.s[0]));                            // before the buffer goes back to the pool
  return SSO_OK;
}

// pass 1, part r of vector v: gather x[r::P], check it (check != CHECK_NO), size-M FFT, part twiddle, copy to the output rows r M ..
inline int parts_part(Ctx& c, const CurveOps* ops, const CurveSizes& cs, const PartsPlan& pl, const PartsVec& v, uint64_t r, uint32_t check,
                      const char* what, char* err, size_t errcap) {
  const size_t sz = point_size(cs, v.group, 0);
  uint32_t* d_status;
  uint8_t *d_x, *d_y;
  int rc;
  if ((rc = status_buffer(c, &d_status, 0, false, err, errcap))) return rc;
  if ((rc = c.alloc((void**)&d_x, pl.M * sz))) return rc;
  if ((rc = c.alloc((void**)&d_y, pl.M * sz))) return rc;
  if ((rc = gather_h2d(c, v.in + r * sz, pl.P * sz, sz, pl.M, d_x, err, errcap))) return rc;
  // CheckForCorrectness as the transform in one piece applies it: re-encoded in place
  if (check != CHECK_NO && (rc = ops->reencode(c, 0, v.group, d_x, 0, pl.M, d_x, 0, check, 1, nullptr, d_status, err, errcap))) return rc;
  const size_t mark = c.allocs.size();
  if ((rc = ops->group_fft(c, 0, v.group, d_x, pl.log_m - pl.log_p, pl.root, pl.two_adicity, nullptr, d_y, 0, d_status, err, errcap))) return rc;
  c.release(mark);
  if (r != 0 || pl.scale) {
    // Z_r[c] = scale w^(r c) Y_r[c]: tau = w^r from index 0, w = root^(2^(two_adicity - log m)) of order m
    uint32_t* d_table;
    if ((rc = ops->fft_part_tables(c, 0, pl.root, pl.two_adicity - pl.log_m, r, pl.scale, &d_table, err, errcap))) return rc;
    VecBatch b;
    memset(&b, 0, sizeof b);
    b.seg[0].in = d_y; b.seg[0].out = d_y; b.seg[0].n = (uint32_t)pl.M; b.seg[0].has_coeff = pl.scale ? 1 : 0;
    b.nseg = 1; b.total = (uint32_t)pl.M;
    if ((rc = ops->batch_exp(c, 0, v.group, b, 0, d_table, 0, CHECK_NO, d_status, err, errcap))) return rc;
  }
  CUDA_TRY(cudaMemcpyAsync(v.out + r * pl.M * sz, d_y, pl.M * sz, cudaMemcpyDeviceToHost, c.s[0]));
  CUDA_TRY(cudaStreamSynchronize(c.s[0]));
  return parts_status(d_status, what, v.vec, r, pl.P, err, errcap);
}

// pass 2, block blk of vector v: the P-point FFT over the rows r M + [c0, c0 + B) of the output, in place
inline int parts_block(Ctx& c, const CurveOps* ops, const CurveSizes& cs, const PartsPlan& pl, const PartsVec& v, uint64_t blk, const char* what,
                       char* err, size_t errcap) {
  const size_t sz = point_size(cs, v.group, 0), run = pl.B * sz;
  const uint64_t P = pl.P, c0 = blk * pl.B;
  uint32_t* d_status;
  uint8_t* buf[2];
  int rc;
  if ((rc = status_buffer(c, &d_status, 0, false, err, errcap))) return rc;
  for (auto& b : buf)
    if ((rc = c.alloc((void**)&b, P * run))) return rc;
  for (uint64_t r = 0; r < P; r++)
    CUDA_TRY(cudaMemcpyAsync(buf[0] + r * run, v.out + (r * pl.M + c0) * sz, run, cudaMemcpyHostToDevice, c.s[0]));
  int cur = 0;
  for (uint32_t s = 0; s < pl.log_p; s++) {
    const size_t mark = c.allocs.size();
    if ((rc = ops->fft_row_stage(c, 0, v.group, buf[cur], P, pl.B, s, pl.root, pl.two_adicity, d_status, buf[cur ^ 1], err, errcap))) return rc;
    c.release(mark);
    cur ^= 1;
  }
  for (uint64_t r = 0; r < P; r++)
    CUDA_TRY(cudaMemcpyAsync(v.out + (r * pl.M + c0) * sz, buf[cur] + r * run, run, cudaMemcpyDeviceToHost, c.s[0]));
  CUDA_TRY(cudaStreamSynchronize(c.s[0]));
  return parts_status(d_status, what, v.vec, c0, 1, err, errcap);
}

// Both passes over the workers of Pt (one context each; stream.cuh run_pieces: the first failure wins, no further task starts and
// every worker is joined).  Pass 1 deals the parts vector by vector in the order given (the costlier G2 vector first), then the
// `extra` tasks (extra_task(i, ...)); pass 2 the column blocks.
inline int parts_fft(const CurveOps* ops, const CurveSizes& cs, const PartsPlan& pl, const PartsVec* vecs, size_t nvec, const Participants& Pt,
                     uint32_t check, const char* what, size_t extra, const std::function<int(size_t, Ctx&, char*, size_t)>& extra_task,
                     char* err, size_t errcap) {
  int rc = run_pieces(nvec * pl.P + extra, Pt, 1, 1, err, errcap, [&](size_t i, int, Ctx& c, char* e, size_t ec) -> int {
    if (i >= nvec * pl.P) return extra_task(i - nvec * pl.P, c, e, ec);
    return parts_part(c, ops, cs, pl, vecs[i / pl.P], i % pl.P, check, what, e, ec);
  });
  if (rc || pl.P == 1) return rc;
  const uint64_t nb = pl.M / pl.B;
  return run_pieces(nvec * nb, Pt, 1, 1, err, errcap, [&](size_t i, int, Ctx& c, char* e, size_t ec) -> int {
    return parts_block(c, ops, cs, pl, vecs[i / nb], i % nb, what, e, ec);
  });
}

// prepare_phase2 in parts over the devices of this process (not cooperative over a process group): the four coefficient vectors by
// parts_fft, h_g1 in pieces of at most M (its upper inputs tauG1[m .. 2m - 1) checked there; the lower ones are the parts of tauG1),
// and the three single elements checked and re-encoded as in the transform in one piece
inline int p2_prepare_devices(const CurveOps* ops, const P1Layout& L, const FftDomain& d, int log_m, const uint8_t* acc, uint8_t* out,
                              const int* devices, int ndev, int device, char* err, size_t errcap) {
  Participants Pt;
  int rc = resolve_participants(devices, ndev, device, false, Pt, err, errcap);
  if (rc) return rc;
  const CurveSizes& cs = L.cs;
  const uint64_t m = 1ull << log_m;
  uint32_t log_p;
  if ((rc = choose_parts((uint32_t)log_m, std::max(cs.g1u, cs.g2u), Pt, log_p, err, errcap))) return rc;
  const std::vector<uint8_t> minv = fft_inv_size(d, (uint32_t)log_m, ops->fr_bytes);
  const PartsPlan pl = parts_plan((uint32_t)log_m, log_p, d.root_inv, d.two_adicity, minv.data());
  const size_t g1 = cs.g1u, g2 = cs.g2u;
  const size_t o_coeffs_g1 = 2 * g1 + g2, o_coeffs_g2 = o_coeffs_g1 + m * g1, o_alpha = o_coeffs_g2 + m * g2, o_beta = o_alpha + m * g1,
               o_h = o_beta + m * g1;
  const PartsVec vecs[4] = {{GROUP_G2, acc + L.off_u[1], out + o_coeffs_g2, 1}, {GROUP_G1, acc + L.off_u[0], out + o_coeffs_g1, 0},
                            {GROUP_G1, acc + L.off_u[2], out + o_alpha, 2}, {GROUP_G1, acc + L.off_u[3], out + o_beta, 3}};
  const uint64_t nh = (m - 1 + pl.M - 1) / pl.M;
  auto extra = [&](size_t i, Ctx& c, char* err, size_t errcap) -> int {
    uint32_t* d_status;
    int rc2;
    if ((rc2 = status_buffer(c, &d_status, 0, false, err, errcap))) return rc2;
    if (i < nh) {
      // h_g1[i0 + k] = tauG1[m + i0 + k] - tauG1[i0 + k]
      const uint64_t i0 = i * pl.M, cnt = std::min(pl.M, m - 1 - i0);
      const uint8_t* tg1 = acc + L.off_u[0];
      uint8_t *d_lo, *d_hi, *d_h;
      if ((rc2 = c.alloc((void**)&d_lo, cnt * g1))) return rc2;
      if ((rc2 = c.alloc((void**)&d_hi, cnt * g1))) return rc2;
      if ((rc2 = c.alloc((void**)&d_h, cnt * g1))) return rc2;
      CUDA_TRY(cudaMemcpyAsync(d_lo, tg1 + i0 * g1, cnt * g1, cudaMemcpyHostToDevice, c.s[0]));
      CUDA_TRY(cudaMemcpyAsync(d_hi, tg1 + (m + i0) * g1, cnt * g1, cudaMemcpyHostToDevice, c.s[0]));
      if ((rc2 = ops->reencode(c, 0, GROUP_G1, d_hi, 0, cnt, d_hi, 0, CHECK_FULL, 1, nullptr, d_status, err, errcap))) return rc2;
      if ((rc2 = ops->points_sub(c, 0, GROUP_G1, d_hi, d_lo, cnt, d_h, 0, err, errcap))) return rc2;
      CUDA_TRY(cudaMemcpyAsync(out + o_h + i0 * g1, d_h, cnt * g1, cudaMemcpyDeviceToHost, c.s[0]));
      CUDA_TRY(cudaStreamSynchronize(c.s[0]));
      return parts_status(d_status, "accumulator", 0, m + i0, 1, err, errcap);
    }
    // alpha_g1 = alphaTauG1[0], beta_g1 = betaTauG1[0], beta_g2 = betaG2
    static const uint32_t vec[3] = {2, 3, 4}, grp[3] = {GROUP_G1, GROUP_G1, GROUP_G2};
    const size_t o_single[3] = {0, g1, 2 * g1};
    for (int k = 0; k < 3; k++) {
      const size_t sz = point_size(cs, grp[k], 0);
      uint8_t* d_p;
      if ((rc2 = c.alloc((void**)&d_p, sz))) return rc2;
      CUDA_TRY(cudaMemcpyAsync(d_p, acc + L.off_u[vec[k]], sz, cudaMemcpyHostToDevice, c.s[0]));
      if ((rc2 = ops->reencode(c, 0, grp[k], d_p, 0, 1, d_p, 0, CHECK_FULL, 1, nullptr, d_status, err, errcap))) return rc2;
      CUDA_TRY(cudaMemcpyAsync(out + o_single[k], d_p, sz, cudaMemcpyDeviceToHost, c.s[0]));
      CUDA_TRY(cudaStreamSynchronize(c.s[0]));
      if ((rc2 = parts_status(d_status, "accumulator", vec[k], 0, 1, err, errcap))) return rc2;
    }
    return SSO_OK;
  };
  return parts_fft(ops, cs, pl, vecs, 4, Pt, CHECK_FULL, "accumulator", nh + 1, extra, err, errcap);
}

}  // namespace sso
