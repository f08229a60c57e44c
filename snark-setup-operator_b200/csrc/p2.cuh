// Phase-2 (Groth16 MPC) contribution and verification on the parameter container, host side
// (SURVEY.md §8a rows a10, a11; Appendix A.5).  Reference call sites: phase2_cli::contribute::<P> at
// src/bin/contribute.rs:827-838, src/bin/verify_transcript.rs:698-715, src/bin/control.rs:810-824; phase2_cli::verify::<P> at
// src/bin/contribute.rs:990-1007, src/bin/verify_transcript.rs:486-503, 655-672; MPCParameters::read_fast at
// src/bin/get_keys.rs:81-88.
//
// [UP] The container is the `phase2::MPCParameters` serialisation of nimiq/snark-setup @ bd530da over ark-groth16 0.4 /
// ark-serialize 0.4 as recalled (not verifiable in the build image; tests/golden/REFERENCE_RECIPE.md is the way to pin it):
//
//   ProvingKey   vk.alpha_g1 G1 | vk.beta_g2 G2 | vk.gamma_g2 G2 | vk.delta_g2 G2 | vk.gamma_abc_g1 Vec<G1>
//                | beta_g1 G1 | delta_g1 G1 | a_query Vec<G1> | b_g1_query Vec<G1> | b_g2_query Vec<G2> | h_query Vec<G1> | l_query Vec<G1>
//   cs_hash      64 bytes
//   contributions  u32 big-endian count, then per contribution (always uncompressed):
//                delta_after G1 | s G1 | s_delta G1 | r_delta G2 | transcript 64 bytes
//   Vec<T> = u64 little-endian length + elements; points compressed or uncompressed as a whole (challenge files are
//   uncompressed, responses compressed — the phase-1 convention of the same CLI).
//
// contribute:  delta <- Fr::rand(rng); s <- G1::rand(rng); s_delta = delta s;
//              transcript = Blake2b-512(cs_hash || contributions so far (as serialised) || s || s_delta);
//              r = hash_to_g2(transcript); r_delta = delta r; delta_after = delta delta_g1;
//              h_query, l_query *= delta^-1; delta_g1, vk.delta_g2 *= delta; the public key is appended.
// verify:      structure and untouched elements equal; transcript recomputed; same_ratio((s, s_delta), (r, r_delta));
//              delta_after = delta_g1'; same_ratio((delta_g1, delta_g1'), (r, r_delta)); same_ratio((delta_g1, delta_g1'),
//              (delta_g2, delta_g2')); same_ratio(merge_pairs(h, h'), (delta_g2', delta_g2)); the same for l.
#pragma once

namespace sso {

struct P2Vec { size_t off = 0; uint64_t n = 0; uint32_t group = 0; };      // off: first element (after the length prefix)
struct P2View {
  bool compressed = false;
  size_t g1 = 0, g2 = 0;                 // element sizes in this encoding
  size_t alpha_g1 = 0, beta_g2 = 0, gamma_g2 = 0, delta_g2 = 0, beta_g1 = 0, delta_g1 = 0;
  P2Vec gamma_abc, a_query, b_g1_query, b_g2_query, h_query, l_query;
  size_t cs_hash = 0, contrib_count = 0, contribs = 0, end = 0;
  uint32_t n_contrib = 0;
  size_t contrib_size = 0;               // bytes of one serialised public key
};

inline uint64_t rd_u64le(const uint8_t* p) { uint64_t v; memcpy(&v, p, 8); return v; }
inline void wr_u64le(uint8_t* p, uint64_t v) { memcpy(p, &v, 8); }
inline uint32_t rd_u32be(const uint8_t* p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }
inline void wr_u32be(uint8_t* p, uint32_t v) { p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v; }

inline int p2_parse(const uint8_t* buf, size_t len, bool compressed, const CurveSizes& cs, P2View& v, char* err, size_t errcap) {
  v.compressed = compressed;
  v.g1 = point_size(cs, GROUP_G1, compressed);
  v.g2 = point_size(cs, GROUP_G2, compressed);
  v.contrib_size = 3 * cs.g1u + cs.g2u + 64;
  size_t o = 0;
  auto need = [&](size_t n) { return o + n <= len; };
  auto elem = [&](size_t& field, size_t sz) { if (!need(sz)) return false; field = o; o += sz; return true; };
  auto vec = [&](P2Vec& f, uint32_t group) {
    if (!need(8)) return false;
    f.n = rd_u64le(buf + o); o += 8;
    f.off = o; f.group = group;
    const size_t sz = point_size(cs, group, compressed);
    if (f.n > (len - o) / sz) return false;
    o += f.n * sz;
    return true;
  };
  bool ok = elem(v.alpha_g1, v.g1) && elem(v.beta_g2, v.g2) && elem(v.gamma_g2, v.g2) && elem(v.delta_g2, v.g2) && vec(v.gamma_abc, GROUP_G1) &&
            elem(v.beta_g1, v.g1) && elem(v.delta_g1, v.g1) && vec(v.a_query, GROUP_G1) && vec(v.b_g1_query, GROUP_G1) &&
            vec(v.b_g2_query, GROUP_G2) && vec(v.h_query, GROUP_G1) && vec(v.l_query, GROUP_G1) && elem(v.cs_hash, 64) && elem(v.contrib_count, 4);
  if (ok) {
    v.n_contrib = rd_u32be(buf + v.contrib_count);
    v.contribs = o;
    ok = v.n_contrib <= (len - o) / v.contrib_size;
    o += (size_t)v.n_contrib * v.contrib_size;
  }
  if (!ok || o != len) { set_err(err, errcap, "phase-2 parameters: malformed container (%zu bytes, parsed %zu)", len, o); return SSO_E_INPUT; }
  v.end = o;
  return SSO_OK;
}

// size of the container with the element counts of `v` in the other encoding and `extra` more contributions
inline size_t p2_size(const P2View& v, const CurveSizes& cs, bool compressed, uint32_t extra) {
  const size_t g1 = point_size(cs, GROUP_G1, compressed), g2 = point_size(cs, GROUP_G2, compressed);
  uint64_t n1 = v.gamma_abc.n + v.a_query.n + v.b_g1_query.n + v.h_query.n + v.l_query.n;
  return (3 + n1) * g1 + (3 + v.b_g2_query.n) * g2 + 6 * 8 + 64 + 4 + (size_t)(v.n_contrib + extra) * v.contrib_size;
}

// the elements of a container in file order: (offset, count, group); single elements have count 1
struct P2Item { size_t off; uint64_t n; uint32_t group; int len_prefix; int kind; };   // kind: 0 untouched, 1 h/l query, 2 delta_g1, 3 delta_g2
inline std::vector<P2Item> p2_items(const P2View& v) {
  return {{v.alpha_g1, 1, GROUP_G1, 0, 0}, {v.beta_g2, 1, GROUP_G2, 0, 0}, {v.gamma_g2, 1, GROUP_G2, 0, 0}, {v.delta_g2, 1, GROUP_G2, 0, 3},
          {v.gamma_abc.off, v.gamma_abc.n, GROUP_G1, 1, 0}, {v.beta_g1, 1, GROUP_G1, 0, 0}, {v.delta_g1, 1, GROUP_G1, 0, 2},
          {v.a_query.off, v.a_query.n, GROUP_G1, 1, 0}, {v.b_g1_query.off, v.b_g1_query.n, GROUP_G1, 1, 0},
          {v.b_g2_query.off, v.b_g2_query.n, GROUP_G2, 1, 0}, {v.h_query.off, v.h_query.n, GROUP_G1, 1, 1}, {v.l_query.off, v.l_query.n, GROUP_G1, 1, 1}};
}

// transcript = Blake2b-512(cs_hash || contributions so far || s || s_delta)
inline void p2_transcript(const uint8_t* buf, const P2View& v, const uint8_t* s_pair, size_t g1u, uint8_t out[64]) {
  Blake2b h(64);
  h.update(buf + v.cs_hash, 64);
  h.update(buf + v.contribs, (size_t)v.n_contrib * v.contrib_size);
  h.update(s_pair, 2 * g1u);
  h.final(out, 64);
}

// One pass over the elements of `in` (view vi) into `out` (view layout vo, same counts): every group re-encoded on the
// device; with delta (contribute) the h / l queries are multiplied by delta^-1 and delta_g1 / delta_g2 by delta.
//   delta == nullptr: plain re-encoding with the given checks (verification: response -> new challenge)
inline int p2_transform(Ctx& c, const CurveOps* ops, const CurveSizes& cs, const uint8_t* in, const P2View& vi, uint8_t* out, bool out_compressed,
                        const uint8_t* delta, const uint8_t* delta_inv, uint32_t check, uint32_t subgroup, const char* what, char* err,
                        size_t errcap) {
  int rc;
  std::vector<P2Item> items = p2_items(vi);
  size_t o = 0;
  std::vector<uint8_t> one(ops->fr_bytes, 0);
  one[0] = 1;
  uint32_t* d_status;
  if ((rc = status_buffer(c, &d_status, 0, false, err, errcap))) return rc;
  const uint64_t SEG = 1ull << 22;
  for (const P2Item& it : items) {
    const size_t isz = point_size(cs, it.group, vi.compressed), osz = point_size(cs, it.group, out_compressed);
    if (it.len_prefix) { wr_u64le(out + o, it.n); o += 8; }
    for (uint64_t lo = 0; lo < it.n; lo += SEG) {
      uint64_t cnt = it.n - lo < SEG ? it.n - lo : SEG;
      uint8_t *d_in, *d_out;
      if ((rc = c.alloc((void**)&d_in, cnt * isz))) return rc;
      if ((rc = c.alloc((void**)&d_out, cnt * osz))) return rc;
      CUDA_TRY(cudaMemcpyAsync(d_in, in + it.off + lo * isz, cnt * isz, cudaMemcpyHostToDevice, c.s[0]));
      const uint8_t* scalar = !delta ? nullptr : (it.kind == 1 ? delta_inv : (it.kind == 2 || it.kind == 3) ? delta : nullptr);
      if (scalar) {
        const uint8_t* coeffs[TAU_COEFF_SLOTS] = {scalar, nullptr, nullptr};
        uint32_t* d_table;
        if ((rc = ops->tau_tables(c, 0, 0, one.data(), coeffs, &d_table, err, errcap))) return rc;
        VecBatch b;
        memset(&b, 0, sizeof b);
        b.seg[0].in = d_in; b.seg[0].out = d_out; b.seg[0].n = (uint32_t)cnt; b.seg[0].coeff_slot = 0; b.seg[0].has_coeff = 1; b.seg[0].mode = 1;
        b.nseg = 1; b.total = (uint32_t)cnt;
        if (check == CHECK_FULL && (rc = ops->reencode(c, 0, it.group, d_in, vi.compressed, cnt, nullptr, 0, CHECK_FULL, 1, nullptr, d_status, err, errcap))) return rc;
        if ((rc = ops->batch_exp(c, 0, it.group, b, vi.compressed, d_table, out_compressed, check, d_status, err, errcap))) return rc;
      } else {
        if ((rc = ops->reencode(c, 0, it.group, d_in, vi.compressed, cnt, d_out, out_compressed, check, subgroup, nullptr, d_status, err, errcap))) return rc;
      }
      CUDA_TRY(cudaMemcpyAsync(out + o + lo * osz, d_out, cnt * osz, cudaMemcpyDeviceToHost, c.s[0]));
      CUDA_TRY(cudaStreamSynchronize(c.s[0]));
      if ((rc = check_status(c, d_status, what, err, errcap))) return rc;
    }
    o += it.n * osz;
  }
  memcpy(out + o, in + vi.cs_hash, 64 + 4 + (size_t)vi.n_contrib * vi.contrib_size);
  return SSO_OK;
}

}  // namespace sso
