/* sso_b200 — C ABI of the B200-native compute core for the phase-1 / phase-2 hot path of
 * nimiq/snark-setup-operator.
 *
 * Drop-in boundary (SURVEY.md §8b): the operator's binaries call the Rust crates
 *   phase1_cli::contribute                      reference src/bin/contribute.rs:811-823,
 *                                               src/bin/verify_transcript.rs:678-696, src/bin/control.rs:793-808
 *   phase1_cli::transform_pok_and_correctness   src/bin/contribute.rs:968-986, src/bin/verify_transcript.rs:466-484
 *   phase1_cli::transform_ratios                src/bin/verify_transcript.rs:646-653, src/bin/control.rs:587-591
 *   phase1_cli::combine / new_challenge         src/bin/verify_transcript.rs:603-607, src/bin/new_setup.rs:105-109
 *   phase2_cli::contribute::<P>                 src/bin/contribute.rs:827-838
 * with file names (or mmapped byte buffers underneath) as arguments and panic on failure.
 * Every export below is what a Rust `-sys` crate (bindgen) binds in their place; INTEGRATION.md
 * shows the shim.  Plain pointers and sizes only; no C++ or torch types.
 *
 * Conventions
 *   - return value: 0 = ok, negative = error class (SSO_E_*); a human-readable message is
 *     written to `err` (NUL-terminated, at most errcap bytes) — the Rust shim turns non-zero into
 *     `panic!("{err}")`, which is the reference's error convention (src/bin/contribute.rs:842-856).
 *   - a failed verification is an error return (SSO_E_VERIFY), not a separate boolean.
 *   - scalars are canonical little-endian byte strings of the curve's Fr size (32/48/95/95).
 *   - `_dev` entry points take DEVICE pointers (inputs already resident in HBM) and enqueue on
 *     internal streams, returning after the work completed; `_buf` take HOST pointers and do
 *     the copies themselves; `_file` take paths, mirroring the reference signatures.
 *   - every call is re-entrant (own streams, stream-ordered scratch), so raising the
 *     operator's --max-in-process-lane to the GPU count shards chunks with no other change.
 *   - there is NO CPU fallback: without a CUDA device every compute entry returns SSO_E_CUDA.
 */
#ifndef SSO_B200_H
#define SSO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* curveKind (reference src/data_structs.rs:123-131; "bw6" default at src/bin/new_setup.rs:53-54) */
enum { SSO_CURVE_BLS12_377 = 0, SSO_CURVE_BW6_761 = 1, SSO_CURVE_MNT4_753 = 2, SSO_CURVE_MNT6_753 = 3 };
enum { SSO_G1 = 0, SSO_G2 = 1 };
/* setup_utils::CheckForCorrectness (used at src/bin/contribute.rs:816-819, 971-980) */
enum { SSO_CHECK_NO = 0, SSO_CHECK_NONZERO = 1, SSO_CHECK_FULL = 2 };
/* setup_utils::SubgroupCheckMode (src/bin/contribute.rs:38-43; verify_transcript.rs:461-464) */
enum { SSO_SUBGROUP_AUTO = 0, SSO_SUBGROUP_DIRECT = 1, SSO_SUBGROUP_BATCHED = 2, SSO_SUBGROUP_NO = 3 };
/* setup_utils::BatchExpMode — accepted and ignored: outputs are mode-independent */
enum { SSO_BATCHEXP_AUTO = 0, SSO_BATCHEXP_DIRECT = 1, SSO_BATCHEXP_BATCH_INVERSION = 2 };
/* phase1::ContributionMode / ProvingSystem (src/utils.rs:326-352) */
enum { SSO_MODE_CHUNKED = 0, SSO_MODE_FULL = 1 };
enum { SSO_PROVING_GROTH16 = 0, SSO_PROVING_MARLIN = 1 };

enum {
  SSO_OK = 0,
  SSO_E_ARG = -1,      /* invalid argument / size mismatch (the reference asserts file lengths) */
  SSO_E_CUDA = -2,     /* CUDA runtime error or no device */
  SSO_E_INPUT = -3,    /* input failed its correctness check (non-canonical, not on curve, zero, ...) */
  SSO_E_VERIFY = -4,   /* verification verdict: reject */
  SSO_E_IO = -5        /* file could not be read / created (outputs are created with O_EXCL) */
};

/* phase1::Phase1Parameters as built by create_parameters_for_chunk / create_full_parameters
 * (reference src/utils.rs:326-352). */
typedef struct {
  uint32_t curve;
  uint32_t proving_system;
  uint32_t contribution_mode;
  uint32_t power;
  uint64_t chunk_index;
  uint64_t chunk_size;
  uint64_t batch_size;
} sso_p1_params_t;

/* indices into the array filled by sso_p1_sizes */
enum {
  SSO_SZ_POWERS_LENGTH = 0, SSO_SZ_POWERS_G1_LENGTH = 1, SSO_SZ_G1_COUNT = 2, SSO_SZ_OTHER_COUNT = 3,
  SSO_SZ_ACCUMULATOR = 4,   /* challenge file size (uncompressed)          */
  SSO_SZ_CONTRIBUTION = 5,  /* response file size (compressed + public key) */
  SSO_SZ_PUBLIC_KEY = 6, SSO_SZ_NUM_CHUNKS = 7
};

const char* sso_version(void);
/* number of usable CUDA devices (0 if none) */
int32_t sso_device_count(void);
/* name of device `device` (e.g. "NVIDIA B200") for ContributedData.processor_data (src/bin/contribute.rs:858-864) */
int32_t sso_device_name(int device, char* out, size_t cap);

/* Phase1Parameters size arithmetic (host only). Replaces the accumulator_size / contribution_size /
 * powers_length fields read at reference src/utils.rs:526-532, src/bin/new_setup.rs:95-102, 265-277. */
int32_t sso_p1_sizes(const sso_p1_params_t* p, uint64_t out[8], char* err, size_t errcap);
/* serialized element sizes: out = {g1 compressed, g1 uncompressed, g2 compressed, g2 uncompressed, Fr bytes} */
int32_t sso_curve_sizes(uint32_t curve, uint64_t out[5]);

/* setup_utils::batch_exp on one vector (K1-K4): out[j] = (coeff * tau^(first_index + j)) * in[j].
 * d_in / d_out are device pointers to n serialized points; coeff may be NULL (= 1). */
int32_t sso_batch_exp_dev(uint32_t curve, uint32_t group, const void* d_in, uint32_t in_compressed, uint64_t n,
                          uint64_t first_index, const uint8_t* tau, const uint8_t* coeff, void* d_out,
                          uint32_t out_compressed, uint32_t check_input, int device, char* err, size_t errcap);

/* phase-2 batch_mul (K7): out[j] = scalar * in[j] for one shared scalar (delta^-1 for the H / L queries,
 * reference src/bin/contribute.rs:827-838). */
int32_t sso_batch_mul_dev(uint32_t curve, uint32_t group, const void* d_in, uint32_t in_compressed, uint64_t n,
                          const uint8_t* scalar, void* d_out, uint32_t out_compressed, uint32_t check_input,
                          int device, char* err, size_t errcap);

/* read_batch + write_batch alone: re-encode n points between the compressed and uncompressed formats
 * with the correctness / subgroup checks of transform_pok_and_correctness and combine. */
int32_t sso_reencode_dev(uint32_t curve, uint32_t group, const void* d_in, uint32_t in_compressed, uint64_t n,
                         void* d_out, uint32_t out_compressed, uint32_t check, uint32_t subgroup_check,
                         int device, char* err, size_t errcap);

/* setup_utils::power_pairs (K3 + K5): decode and check n points, draw scalars r_i, return the pair
 * (sum r_i v_i, sum r_i v_{i+1}) over i < n-1 as two uncompressed points in out_pair (host).  The reference
 * draws r_i from thread_rng, so only the verdict downstream is comparable; seed32 == NULL uses fresh host
 * entropy, a 32-byte seed makes the scalars reproducible (tests): r_i = first 120 bits of the ChaCha20(seed32)
 * keystream block 2i (uniform 120-bit scalars: soundness error 2^-120, a third to a sixth of the work of full-size ones).  TEST-ONLY: two MSMs run with the same seed share their r_i, which
 * makes a G1-vs-G2 comparison of their results vacuous; the verification flows (sso_p1_verify_chunk_*, sso_p1_verify_ratios_file,
 * sso_p2_verify_queries_buf) derive a distinct ChaCha20 key per MSM, Blake2b-256(seed || vector id || chunk || piece || rank). */
int32_t sso_power_pairs_dev(uint32_t curve, uint32_t group, const void* d_in, uint32_t in_compressed, uint64_t n,
                            uint32_t check, uint32_t subgroup_check, const uint8_t* seed32, uint8_t* out_pair, size_t out_len,
                            int device, char* err, size_t errcap);
/* setup_utils::merge_pairs: (sum r_i a_i, sum r_i b_i) for two vectors of n points (same conventions). */
int32_t sso_merge_pairs_dev(uint32_t curve, uint32_t group, const void* d_a, const void* d_b, uint32_t in_compressed, uint64_t n,
                            uint32_t check, uint32_t subgroup_check, const uint8_t* seed32, uint8_t* out_pair, size_t out_len,
                            int device, char* err, size_t errcap);

/* setup_utils::same_ratio / check_same_ratio (K8) for n checks on HOST buffers.  Check i occupies
 * 2 * |G1 uncompressed| + 2 * |G2 uncompressed| bytes laid out a | b | c | d and asks e(a, d) == e(b, c);
 * verdicts[i] = 1 (same ratio) or 0.  Undecodable or off-curve inputs are SSO_E_INPUT. */
int32_t sso_same_ratio(uint32_t curve, const uint8_t* checks, uint64_t n, uint32_t* verdicts, int device, char* err,
                       size_t errcap);

/* Phase1::computation for one chunk, device-resident: d_challenge holds the challenge file image
 * (accumulator_size bytes, uncompressed), d_response receives the compressed vectors at their
 * response-file offsets (contribution_size bytes; the 64-byte hash slot and the public key tail
 * are left untouched for the host). */
int32_t sso_p1_contribute_dev(const sso_p1_params_t* p, const void* d_challenge, void* d_response,
                              const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta,
                              uint32_t check_input, int device, char* err, size_t errcap);

/* The RNG-free core of phase1_cli::contribute on host buffers: copies the challenge to the device,
 * computes, copies the response back, writes Blake2b-512(challenge) into response[0..64) and the
 * caller-supplied serialized public key into the tail. */
int32_t sso_p1_contribute_buf(const sso_p1_params_t* p, const uint8_t* challenge, size_t challenge_len,
                              uint8_t* response, size_t response_len, const uint8_t* tau, const uint8_t* alpha,
                              const uint8_t* beta, const uint8_t* pubkey, size_t pubkey_len, uint32_t check_input,
                              int device, char* err, size_t errcap);

/* sso_p1_contribute_buf over several chunks in flight, as the reference's Process lane holds several chunks
 * (src/bin/contribute.rs:64-71, 158-163: --max-in-process-lane; chunks are independent, :1132-1139).
 * params[i], challenges[i], responses[i] describe chunk i; the same scalars and public key are applied to all.
 * host_threads workers (0 = default: 3 per device) each run one chunk at a time on their own CUDA streams: the
 * sequential Blake2b of one chunk overlaps the copies and kernels of the others.  device < 0 spreads the workers
 * over all visible devices (worker t on device t mod count).  Results are byte-identical to n_chunks separate
 * sso_p1_contribute_buf calls.  On failure the first error is returned and no further chunks start. */
int32_t sso_p1_contribute_many_buf(const sso_p1_params_t* params, size_t n_chunks, const uint8_t* const* challenges,
                                   const size_t* challenge_lens, uint8_t* const* responses, const size_t* response_lens,
                                   const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta, const uint8_t* pubkey,
                                   size_t pubkey_len, uint32_t check_input, uint32_t host_threads, int device, char* err,
                                   size_t errcap);

/* sso_p1_contribute_seeded_buf (all of phase1_cli::contribute but the file I/O) over several chunks in flight: the
 * contributor applies the same seed-derived key to every chunk (src/bin/contribute.rs:789, 809-823).  Worker / device
 * semantics as sso_p1_contribute_many_buf. */
int32_t sso_p1_contribute_seeded_many_buf(const sso_p1_params_t* params, size_t n_chunks, const uint8_t* const* challenges,
                                          const size_t* challenge_lens, uint8_t* const* responses, const size_t* response_lens,
                                          const uint8_t seed32[32], uint32_t check_input, uint32_t host_threads, int device,
                                          char* err, size_t errcap);

/* sso_p1_verify_chunk_buf over several chunks in flight: the chunk loop of verify_transcript
 * (src/bin/verify_transcript.rs:293-569) as a work queue.  Same worker / device semantics as
 * sso_p1_contribute_many_buf; the first failing chunk's code and message are returned (SSO_E_VERIFY names the check). */
int32_t sso_p1_verify_chunk_many_buf(const sso_p1_params_t* params, size_t n_chunks, const uint8_t* const* challenges,
                                     const size_t* challenge_lens, const uint8_t* const* responses, const size_t* response_lens,
                                     uint8_t* const* new_challenges, const size_t* new_challenge_lens, uint32_t check_input,
                                     uint32_t check_output, uint32_t subgroup_check_mode, uint32_t ratio_check,
                                     const uint8_t* rlc_seed32, uint32_t host_threads, int device, char* err, size_t errcap);

/* phase1_cli::new_challenge (reference src/bin/new_setup.rs:105-109, src/bin/verify_transcript.rs:322-326):
 * the initial accumulator — every element is the group generator, hash slot = Blake2b-512 of the empty
 * string.  d_challenge: accumulator_size bytes on the device.  NOTE: for MNT4-753 / MNT6-753 G2 the
 * arkworks generator constant is not recoverable in this environment; a derived order-r point stands
 * in (DESIGN.md "known gaps"). */
int32_t sso_p1_new_challenge_dev(const sso_p1_params_t* p, void* d_challenge, int device, char* err, size_t errcap);

/* Kernel accounting.  Launch counts are always kept; with profiling enabled every kernel launch is
 * bracketed by CUDA events on its own stream.  sso_profile_read fills (launches, nanoseconds, elements)
 * triples per kernel kind, in the order of SSO_PK_*, and returns the number of kinds.  sso_profile_enable(2)
 * additionally runs every call on a single stream, so that a kernel's event time is its time alone on the GPU. */
enum { SSO_PK_TAU_TABLES = 0, SSO_PK_BATCH_EXP_G1, SSO_PK_BATCH_EXP_G2, SSO_PK_NORMALIZE_G1, SSO_PK_NORMALIZE_G2,
       SSO_PK_REENCODE_G1, SSO_PK_REENCODE_G2, SSO_PK_FILL, SSO_PK_MSM, SSO_PK_OTHER, SSO_PK_BATCH_EXP_CHUNK,
       SSO_PK_NORMALIZE_CHUNK, SSO_PK_COUNT };
int32_t sso_profile_enable(int32_t on);
int32_t sso_profile_reset(void);
int32_t sso_profile_read(uint64_t* out, size_t cap);

/* Phase1::key_generation (reached from phase1_cli::contribute, reference src/bin/contribute.rs:789, 811-823): the
 * contributor RNG is ChaCha20 seeded with seed32 (setup_utils::derive_rng_from_seed); digest64 = Blake2b(challenge).
 * scalars_out: tau | alpha | beta canonical little-endian (3 * Fr bytes); pubkey_out: the serialized PublicKey
 * (tau_g1.0, tau_g1.1, alpha_g1.0, alpha_g1.1, beta_g1.0, beta_g1.1, tau_g2, alpha_g2, beta_g2, all uncompressed). */
int32_t sso_p1_keygen(uint32_t curve, const uint8_t seed32[32], const uint8_t digest64[64], uint8_t* scalars_out, size_t scalars_len,
                      uint8_t* pubkey_out, size_t pubkey_len, int device, char* err, size_t errcap);

/* phase1_cli::contribute on host buffers, including hashing, key generation from the seeded RNG and the public key. */
int32_t sso_p1_contribute_seeded_buf(const sso_p1_params_t* p, const uint8_t* challenge, size_t challenge_len, uint8_t* response,
                                     size_t response_len, const uint8_t seed32[32], uint32_t check_input, int device, char* err,
                                     size_t errcap);

/* phase1_cli::contribute(challenge_fn, challenge_hash_fn, response_fn, response_hash_fn, check_input, batch_exp_mode,
 * &parameters, rng) — reference src/bin/contribute.rs:811-823, src/bin/verify_transcript.rs:678-696,
 * src/bin/control.rs:793-808.  The rng argument becomes its 32-byte seed.  Output files must not exist. */
int32_t sso_p1_contribute_file(const sso_p1_params_t* p, const char* challenge_fn, const char* challenge_hash_fn,
                               const char* response_fn, const char* response_hash_fn, uint32_t check_input, uint32_t batch_exp_mode,
                               const uint8_t seed32[32], int device, char* err, size_t errcap);

/* Phase1::verification of one chunk on host buffers (row a5): hash chain, proofs of knowledge, per-element checks of
 * the response (check_output, subgroup_check_mode), chunk-0 update checks, optional power-ratio checks via random
 * linear combinations (ratio_check), and the decompressed new challenge whose hash slot is Blake2b(response).
 * A rejected contribution is SSO_E_VERIFY with the failed check named in err.  rlc_seed32 == NULL: fresh entropy.
 *   check_input  : CheckForCorrectness applied to the challenge vectors (No: skipped — the operator's default; Full: on the
 *                  curve and in the subgroup)
 *   check_output : every response element must be non-zero whatever the setting; Full also forces the membership test
 *   subgroup_check_mode : Auto / Direct / Batched run the membership test [r]P = O on every response element, No skips it —
 *                  independent of check_output, as in the reference call (src/bin/contribute.rs:971-984)
 *   ratio_check  : power ratios of the chunk's vectors against its tau_g2 combination; a chunk past 2^power holds tau_g1 only
 *                  (no G2 element to compare with): its ratios are covered by sso_p1_verify_ratios_file on the combined file
 * The nine public-key points must be non-zero and in their subgroups.  Full mode (and chunks beyond 2^22 elements) stream the
 * vectors in `batch_size` pieces. */
int32_t sso_p1_verify_chunk_buf(const sso_p1_params_t* p, const uint8_t* challenge, size_t challenge_len, const uint8_t* response,
                                size_t response_len, uint8_t* new_challenge, size_t new_challenge_len, uint32_t check_input,
                                uint32_t check_output, uint32_t subgroup_check_mode, uint32_t ratio_check, const uint8_t* rlc_seed32,
                                int device, char* err, size_t errcap);

/* phase1_cli::transform_pok_and_correctness(challenge_fn, challenge_hash_fn, check_input, response_fn, response_hash_fn,
 * check_output, new_challenge_fn, new_challenge_hash_fn, subgroup_check_mode, ratio_check, &parameters) —
 * reference src/bin/contribute.rs:968-986, src/bin/verify_transcript.rs:466-484, 746-776, src/bin/control.rs:841-865. */
int32_t sso_p1_verify_chunk_file(const sso_p1_params_t* p, const char* challenge_fn, const char* challenge_hash_fn, uint32_t check_input,
                                 const char* response_fn, const char* response_hash_fn, uint32_t check_output,
                                 const char* new_challenge_fn, const char* new_challenge_hash_fn, uint32_t subgroup_check_mode,
                                 uint32_t ratio_check, int device, char* err, size_t errcap);

/* phase1_cli::new_challenge(challenge_fn, challenge_hash_fn, &parameters) — reference src/bin/new_setup.rs:105-109,
 * src/bin/verify_transcript.rs:322-326: the initial accumulator of a chunk (or of the whole ceremony in Full mode): every
 * element the group generator, hash slot = Blake2b-512 of the empty input; writes the file and the 64 raw bytes of its hash.
 * Output files must not exist. */
int32_t sso_p1_new_challenge_file(const char* challenge_fn, const char* challenge_hash_fn, const sso_p1_params_t* p, int device,
                                  char* err, size_t errcap);

/* The generators new_challenge writes and chunk-0 / transform_ratios verification compare against, per curve and process:
 * one uncompressed G1 point and one uncompressed G2 point (checked: non-zero, on the curve, in the order-r subgroup).
 * Built in: arkworks' constants except the G2 generators of MNT4-753 / MNT6-753, which could not be recovered in the build
 * environment and default to a derived point — an integrator hands the reference's over once (e.g. from the round-0
 * challenge the operator regenerates, reference src/bin/verify_transcript.rs:316-361).  Both NULL: back to the built-ins. */
int32_t sso_p1_set_generators(uint32_t curve, const uint8_t* g1_uncompressed, size_t g1_len, const uint8_t* g2_uncompressed,
                              size_t g2_len, int device, char* err, size_t errcap);

/* phase1_cli::combine(response_list_fn, combined_fn, &parameters) — reference src/bin/verify_transcript.rs:603-607,
 * src/bin/control.rs:564-568.  `p`: the chunk-0 parameters of the ceremony, as the reference passes them.  The list file names
 * one response file (compressed + public key) per chunk, one path per line, in chunk order.  Output: the Full-mode accumulator,
 * uncompressed, hash slot zero.  Decoding is streamed in `batch_size` pieces over devices[0..ndev) (NULL / 0: `device`; -1: all). */
int32_t sso_p1_combine_file(const char* response_list_fn, const char* combined_fn, const sso_p1_params_t* p, const int* devices,
                            int ndev, int device, char* err, size_t errcap);

/* phase1_cli::transform_ratios(response_fn, check_input, &parameters) — reference src/bin/verify_transcript.rs:646-653, 811-822,
 * src/bin/control.rs:587-591, 866-873: consistency of a whole uncompressed accumulator (generators in element 0, power ratios of
 * the four vectors by random linear combinations, beta_g2).  The vectors are streamed in `batch_size` pieces over
 * devices[0..ndev) of this process — or over the ranks of the process group (sso_dist_init) —, every participant sums the
 * partial pairs of its pieces, ONE NCCL all-gather exchanges the per-participant sums and a point addition folds them
 * (SURVEY.md §8e).  rlc_seed32 == NULL: fresh entropy (the only sound setting outside tests).  SSO_E_VERIFY on rejection. */
int32_t sso_p1_verify_ratios_file(const sso_p1_params_t* p, const char* combined_fn, uint32_t check_input, const int* devices,
                                  int ndev, int device, const uint8_t* rlc_seed32, char* err, size_t errcap);

/* Process group for the cooperative calls: one process per GPU (torchrun), every rank makes the same call on the same
 * files.  Cooperative are the Full-mode calls (sso_p1_contribute_file / _seeded_buf / sso_p1_verify_chunk_file / _buf with
 * contribution_mode = SSO_MODE_FULL), sso_p1_combine_file and sso_p1_verify_ratios_file: pieces are dealt round-robin over
 * the ranks, outputs are written into the shared file mapping, rank 0 creates and commits the files, and the partial MSM
 * results meet in one ncclAllGather.  Chunk-level calls stay local to the calling rank.
 *   sso_dist_unique_id : ncclGetUniqueId on one rank; the caller broadcasts the 128 bytes (e.g. over torch.distributed)
 *   sso_dist_init      : ncclCommInitRank on `device`;  sso_dist_barrier: all ranks;  sso_dist_finalize: destroys it
 *   sso_dist_stats     : [0] initialised [1] rank [2] world [3] all-gathers issued so far [4] NCCL version code */
int32_t sso_dist_unique_id(uint8_t out[128], char* err, size_t errcap);
int32_t sso_dist_init(int32_t rank, int32_t world, const uint8_t id128[128], int device, char* err, size_t errcap);
int32_t sso_dist_barrier(char* err, size_t errcap);
int32_t sso_dist_finalize(void);
int32_t sso_dist_stats(uint64_t out[5]);

/* Sum of n uncompressed points (host buffers) -> one uncompressed point.  Used to combine the per-GPU partial
 * results of a sharded power_pairs / merge_pairs after the NCCL all-gather (SURVEY.md §8e). */
int32_t sso_points_sum(uint32_t curve, uint32_t group, const uint8_t* points, uint64_t n, uint8_t* out, size_t out_len, int device,
                       char* err, size_t errcap);

/* phase2_cli::contribute core (reference src/bin/contribute.rs:827-838; SURVEY.md §8a row a10): multiply every
 * point of a G1 query vector (h_query or l_query) by delta^-1.  Host buffers of n serialized G1 points. */
int32_t sso_p2_scale_queries_buf(uint32_t curve, const uint8_t* in, size_t in_len, uint8_t* out, size_t out_len, uint64_t n,
                                 const uint8_t* delta_inv, uint32_t in_compressed, uint32_t out_compressed, uint32_t check_input,
                                 int device, char* err, size_t errcap);

/* phase2_cli::verify core (reference src/bin/contribute.rs:990-1007; row a11): accepts iff
 * same_ratio(merge_pairs(query_before, query_after), (delta_g2_after, delta_g2_before)); SSO_E_VERIFY otherwise. */
int32_t sso_p2_verify_queries_buf(uint32_t curve, const uint8_t* before, size_t before_len, const uint8_t* after, size_t after_len,
                                  uint64_t n, uint32_t before_compressed, uint32_t after_compressed, const uint8_t* delta_g2_before,
                                  const uint8_t* delta_g2_after, uint32_t check, uint32_t subgroup_check, const uint8_t* rlc_seed32,
                                  int device, char* err, size_t errcap);

/* phase2_cli::contribute::<P> / phase2_cli::verify::<P> on the Groth16 parameter container (rows a10, a11; reference
 * src/bin/contribute.rs:827-838, 990-1007, src/bin/verify_transcript.rs:486-503, 655-672, 698-715, src/bin/control.rs:633-644,
 * 810-824; MPCParameters::read_fast at src/bin/get_keys.rs:81-88).  The curve type parameter becomes `curve`, the rng its
 * 32-byte seed.  Container ([UP] phase2::MPCParameters over ark-groth16 0.4, as recalled — see csrc/p2.cuh):
 *   vk.alpha_g1 | vk.beta_g2 | vk.gamma_g2 | vk.delta_g2 | vk.gamma_abc_g1[] | beta_g1 | delta_g1 | a_query[] | b_g1_query[] |
 *   b_g2_query[] | h_query[] | l_query[] | cs_hash[64] | u32 BE count | contributions (delta_after, s, s_delta, r_delta, transcript)
 * challenge files uncompressed, responses compressed; vectors carry a u64 LE length.
 *   contribute: delta <- Fr::rand, s <- G1::rand; proof of knowledge bound to the transcript of the earlier contributions;
 *               h_query, l_query *= delta^-1 (the batch_mul of K7), delta_g1, vk.delta_g2 *= delta; the public key is appended
 *   verify:     structure and untouched elements equal, transcript chain, proof of knowledge, delta_g1 / delta_g2 updates and
 *               same_ratio(merge_pairs(query_before, query_after), (delta_g2_after, delta_g2_before)) for h and l; writes the
 *               decompressed new challenge.  verify_full is accepted for signature parity (this container is always whole).
 * `_buf`: *out_len receives the size of the output; SSO_E_ARG (with the size) when the capacity is too small. */
int32_t sso_p2_contribute_buf(uint32_t curve, const uint8_t* challenge, size_t challenge_len, uint8_t* response, size_t response_cap,
                              size_t* response_len, const uint8_t seed32[32], uint32_t check_input, int device, char* err, size_t errcap);
int32_t sso_p2_contribute_file(uint32_t curve, const char* challenge_fn, const char* challenge_hash_fn, const char* response_fn,
                               const char* response_hash_fn, uint32_t check_input, uint32_t batch_exp_mode, const uint8_t seed32[32],
                               int device, char* err, size_t errcap);
int32_t sso_p2_verify_buf(uint32_t curve, const uint8_t* challenge, size_t challenge_len, const uint8_t* response, size_t response_len,
                          uint8_t* new_challenge, size_t new_challenge_cap, size_t* new_challenge_len, uint32_t check_input,
                          uint32_t check_output, uint32_t subgroup_check_mode, const uint8_t* rlc_seed32, int device, char* err,
                          size_t errcap);
int32_t sso_p2_verify_file(uint32_t curve, const char* challenge_fn, const char* challenge_hash_fn, uint32_t check_input,
                           const char* response_fn, const char* response_hash_fn, uint32_t check_output, const char* new_challenge_fn,
                           const char* new_challenge_hash_fn, uint32_t subgroup_check_mode, uint32_t verify_full, int device, char* err,
                           size_t errcap);

/* Radix-2 group FFT of 2^log_n points of one group over the scalar field's two-adic domain (ark-poly Radix2EvaluationDomain
 * fft / ifft applied to curve points, the primitive of phase2_cli::prepare_phase2, reference
 * src/bin/intermediate_transform.rs:213-226).  inverse = 0: out_i = sum_j w^(ij) in_j; inverse = 1: out_i = 2^-log_n sum_j w^(-ij) in_j,
 * natural order, w = GENERATOR^((r - 1) / 2^log_n).  log_n is at most the 2-adicity of Fr and 24.  d_out may equal d_in. */
int32_t sso_group_fft_dev(uint32_t curve, uint32_t group, const void* d_in, uint32_t in_compressed, uint32_t log_n, uint32_t inverse,
                          void* d_out, uint32_t out_compressed, int device, char* err, size_t errcap);
/* phase2_cli::prepare_phase2 (reference src/bin/intermediate_transform.rs:213-226) on host buffers: a Full-mode Groth16 accumulator
 * (uncompressed) -> the Lagrange-basis Groth16Params of phase2_size = m points (a power of two, m <= 2^power; MNT6-753: m <= 2^15):
 * alpha_g1 | beta_g1 | beta_g2 | coeffs_g1[m] | coeffs_g2[m] | alpha_coeffs_g1[m] | beta_coeffs_g1[m] | h_g1[m - 1], uncompressed.
 * Every accumulator element read must be non-zero, on the curve and in the subgroup (SSO_E_INPUT otherwise).
 * *out_len receives the size of the output; SSO_E_ARG (with the size) when out_cap is too small. */
int32_t sso_p2_prepare_buf(const sso_p1_params_t* p, const uint8_t* accumulator, size_t len, uint64_t phase2_size, uint8_t* out, size_t out_cap,
                           size_t* out_len, int device, char* err, size_t errcap);
/* phase2_cli::prepare_phase2(phase2_filename, response_filename, phase2_size, parameters), argument for argument; the output must not
 * exist (SSO_E_IO) and is only renamed into place when the call succeeded. */
int32_t sso_p2_prepare_file(const char* phase2_fn, const char* response_fn, uint64_t phase2_size, const sso_p1_params_t* p, int device,
                            char* err, size_t errcap);

/* setup_utils::calculate_hash (reference src/utils.rs:618-623): Blake2b-512, unkeyed. Host only. */
int32_t sso_blake2b_512(const uint8_t* data, size_t len, uint8_t out[64]);

/* Microbenchmark behind roofline.peak: dependent-free 32x32+64 multiply-accumulate chains on all SMs.
 * Returns multiply-accumulates per second (SURVEY.md §8d "IMAD_peak is measured on the box"). */
int32_t sso_imad_peak(int device, int variant, double* macs_per_s, char* err, size_t errcap);

/* Test hook: elementwise field multiplication out[i] = a[i] * b[i] on the device, canonical
 * little-endian elements of the field's serialized size. field: 0 r253, 1 q377, 2 q761, 3 q4(753), 4 q6(753). */
int32_t sso_test_field_mul(uint32_t field, const uint8_t* a, const uint8_t* b, uint8_t* out, uint64_t n, int device,
                           char* err, size_t errcap);
/* Test hook: one field operation per element on raw little-endian Montgomery words, loaded without reduction or range check
 * and returned as the arithmetic leaves them (csrc/field_probe.cuh).  field: 0 r253, 1 q377, 2 q761, 3 q4(753), 4 q6(753),
 * 5 q377^2 (u^2 = -5), 6 q4^2 (u^2 = 13), 7 q6^3 (u^3 = 11), 8-10 the same three extensions over 2 / 3 cooperating lanes.
 * Element i has ops[i] and k[i] (the factor of mad_small_lazy); a, b, out hold n elements of the field's words, coefficient after
 * coefficient.  ops: 0 mul, 1 add, 2 sub, 3 sqr, 4 neg, 5 inv, 6 dedicated sqr, 7 lex_is_neg, 8 sqrt, 9 reduce_small,
 * 10 mad_small_lazy(a, k, b), 11 conj, 12 mul_base(a, b.c0), 13 mul_u2, 14 frob_w.  rc[i]: the predicate of ops 7 / 8 (1 = negative,
 * 1 = root found), 0 otherwise, 0xffffffff for an op the field does not have (out[i] then stays zero). */
int32_t sso_test_field_op(uint32_t field, const uint32_t* ops, const uint32_t* a, const uint32_t* b, const uint32_t* k, uint32_t* out,
                          uint32_t* rc, uint64_t n, int device, char* err, size_t errcap);

#ifdef __cplusplus
}
#endif
#endif /* SSO_B200_H */
