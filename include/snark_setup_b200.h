/*
 * snark_setup_b200.h — C ABI of the B200-native batch-exponentiation engine.
 *
 * This is the drop-in boundary for the ONE hot path of nimiq/snark-setup (SURVEY.md §8): every
 * entry point takes plain pointers and sizes, host memory unless the name ends in `_dev`, and
 * replaces the body of the reference function cited beside it.  The reference has no FFI today;
 * INTEGRATION.md shows the Rust `extern "C"` block + `build.rs` a maintainer adds so that
 * `setup_utils::{batch_exp, batch_mul, generate_powers_of_tau, merge_pairs, power_pairs,
 * check_subgroup}`, `phase1::helpers::buffers::apply_powers` and
 * `phase1::helpers::accumulator::check_*` call into this library.
 *
 * Conventions
 *   - Points cross the boundary in the reference's canonical serialisation (ark-serialize 0.4):
 *     packed elements, no header; `compressed` selects x+flags vs x||y+flags
 *     (sizes: BLS12-377 G1 48/96, G2 96/192; BW6-761 G1 = G2 = 96/192,
 *     phase1/src/objects/parameters.rs:312-317; MNT4-753 G1 95/190, G2 190/380; MNT6-753 G1 95/190, G2 285/570).
 *   - Scalars cross as canonical little-endian integers < r of ss_scalar_size() bytes
 *     (32 for BLS12-377, 48 for BW6-761, 95 for MNT4/6-753) = `Fr::serialize_uncompressed`.
 *   - `check` is setup_utils::CheckForCorrectness (setup-utils/src/elements.rs:18-23).
 *   - Return value: SS_OK or an ss_status error; details of the last error of the calling thread
 *     via ss_last_error().  Errors map 1:1 onto setup_utils::Error (setup-utils/src/errors.rs:11-38).
 *   - The caller owns every buffer; nothing is retained after return; only the bytes of the
 *     output range are written.  Entry points are thread-safe (the reference calls the helpers from
 *     up to 4 rayon tasks at once, phase1/src/computation.rs:68-188).
 *   - There is no CPU fallback: without a usable CUDA device every compute call fails with
 *     SS_ERR_DEVICE.
 */
#ifndef SNARK_SETUP_B200_H
#define SNARK_SETUP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* The curves the reference exposes (setup-utils/src/converters.rs:18-45).  BLS12-377 and BW6-761 are the tuned ceremony
 * curves.  MNT4-753 / MNT6-753 (a != 0, G2 over Fq2 / Fq3, 95-byte field elements) run the same entry points
 * functionally — batch_exp / apply_powers / Phase1::computation, transcode, subgroup checks, merge_pairs / power_pairs,
 * the verification vectors, and prepare_phase2 / QAP evaluation (ss_group_ifft, ss_h_query_groth16,
 * ss_groth16_params_*, ss_qap_dot_product) — without endomorphism speed-ups.  Their radix-2 domains reach 2^30 (MNT4-753
 * Fr) and 2^15 (MNT6-753 Fr); a larger domain fails with SS_ERR_INVALID_ARGUMENT.  Not available for them:
 * ss_phase1_initialization (the arkworks G2 generator constants are not known to this build) and the device pairing
 * checks (ss_*same_ratio*; the (s, sx) pairs are returned for the host's check_same_ratio as SURVEY.md §8 A12 places
 * it). */
typedef enum { SS_CURVE_BLS12_377 = 0, SS_CURVE_BW6_761 = 1, SS_CURVE_MNT4_753 = 2, SS_CURVE_MNT6_753 = 3 } ss_curve;
typedef enum { SS_G1 = 0, SS_G2 = 1 } ss_group;

/* setup_utils::CheckForCorrectness (setup-utils/src/elements.rs:18-23) */
typedef enum { SS_CHECK_FULL = 0, SS_CHECK_ONLY_NON_ZERO = 1, SS_CHECK_ONLY_IN_GROUP = 2, SS_CHECK_NO = 3 } ss_check;
/* setup_utils::SubgroupCheckMode (setup-utils/src/elements.rs:86-91) */
typedef enum { SS_SUBGROUP_AUTO = 0, SS_SUBGROUP_DIRECT = 1, SS_SUBGROUP_BATCHED = 2, SS_SUBGROUP_NO = 3 } ss_subgroup_mode;
/* phase1::ContributionMode / ProvingSystem (phase1/src/objects/parameters.rs) */
typedef enum { SS_MODE_FULL = 0, SS_MODE_CHUNKED = 1 } ss_contribution_mode;
typedef enum { SS_GROTH16 = 0, SS_MARLIN = 1 } ss_proving_system;

typedef enum {
    SS_OK = 0,
    SS_ERR_INVALID_DATA = 1,       /* Error::ZexeSerializationError(InvalidData)      */
    SS_ERR_UNEXPECTED_FLAGS = 2,   /* Error::ZexeSerializationError(UnexpectedFlags)  */
    SS_ERR_POINT_AT_INFINITY = 3,  /* Error::PointAtInfinity                          */
    SS_ERR_INCORRECT_SUBGROUP = 4, /* Error::IncorrectSubgroup                        */
    SS_ERR_INVALID_LENGTH = 5,     /* Error::InvalidLength { expected, got }          */
    SS_ERR_INVALID_CHUNK = 6,      /* Error::InvalidChunk                             */
    SS_ERR_BATCH_TOO_SMALL = 7,    /* Error::BatchTooSmall                            */
    SS_ERR_INVALID_ARGUMENT = 8,   /* (no reference equivalent: bad enum / null pointer)  */
    SS_ERR_DEVICE = 9,             /* CUDA failure; the Rust shim turns this into a panic */
    SS_ERR_INVALID_RATIO = 10      /* VerificationError::InvalidRatio (setup-utils/src/errors.rs:97-100) */
} ss_status;

typedef struct {
    int code;          /* ss_status */
    uint64_t index;    /* element index the error refers to (lowest failing index), or 0 */
    uint64_t expected; /* InvalidLength */
    uint64_t got;      /* InvalidLength */
    char message[160];
} ss_error_info;

/* -------------------------------------------------------------------------------------------- */
/* device management                                                                            */
/* -------------------------------------------------------------------------------------------- */
/* Select the CUDA devices this process uses (n = 0: device 0, or $SNARK_SETUP_GPUS="0,1,.."). */
int ss_init(const int* devices, int n_devices);
void ss_shutdown(void);
int ss_device_count(void);
void ss_last_error(ss_error_info* out);
const char* ss_version(void);

/* Per-kernel timing, the engine's counterpart of the reference's `tracing` spans and its
 * Instant timer around the subgroup loop (phase1/src/computation.rs:26,56;
 * phase1/src/helpers/accumulator.rs:110,140): when enabled, every kernel launch is bracketed by CUDA
 * events on its own stream.  ss_profile_launches() counts launches whether or not timing is on. */
typedef struct {
    char name[64];     /* e.g. "k_scalar_mul<bls12_377.g1>" */
    uint64_t launches; /* kernel launches */
    uint64_t elements; /* group elements processed by those launches */
    double ms;         /* summed device time */
} ss_profile_entry;
void ss_profile_enable(int on);
void ss_profile_reset(void);
uint64_t ss_profile_launches(void);
int ss_profile_read(ss_profile_entry* out, int max_entries);

/* Tuning knob: whether the tau_g1 / tau_g2 / alpha_g1 / beta_g1 / beta_g2 vectors of one
 * ss_phase1_* call are processed concurrently (one internal stream each; default on, or
 * $SS_CONCURRENT_VECTORS=0) — the reference spawns one rayon task per vector the same way
 * (phase1/src/computation.rs:68-188).  Results are identical either way. */
void ss_set_concurrent_vectors(int on);

/* Scalar multiplication of bases that were read WITHOUT a subgroup check (CheckForCorrectness::No / OnlyNonZero —
 * the reference's contribute default, setup-utils/src/helpers.rs:550).  Default (0): the GLV / GLS path, whose
 * result equals the reference's `mul_bigint` for every point of the order-r subgroup — which is what a ceremony's
 * challenge holds, the coordinator having verified it.  1: such bases go through the reference's own MSB-first
 * double-and-add, which reproduces `mul_bigint` on ANY input (off-subgroup, even off-curve) at ~2x the cost.
 * Inputs read with Full / OnlyInGroup always take the fast path. */
void ss_set_strict_unchecked_inputs(int on);

/* buffer_size::<C>(compression) — setup-utils/src/io/mod.rs:13-15 */
size_t ss_element_size(int curve, int group, int compressed);
size_t ss_scalar_size(int curve);

/* -------------------------------------------------------------------------------------------- */
/* setup-utils helpers                                                                          */
/* -------------------------------------------------------------------------------------------- */
/* generate_powers_of_tau — setup-utils/src/helpers.rs:32-37.  out: (end-start) scalars. */
int ss_generate_powers_of_tau(int curve, const uint8_t* tau, uint64_t start, uint64_t end, uint8_t* out);

/* batch_exp — setup-utils/src/helpers.rs:75-140.  `bases`: n uncompressed elements, updated in
 * place; `exps`: n_exps scalars (n_exps != n => SS_ERR_INVALID_LENGTH, helpers.rs:81-86);
 * `coeff`: one scalar or NULL. */
int ss_batch_exp(int curve, int group, uint8_t* bases, size_t n, const uint8_t* exps, size_t n_exps,
                 const uint8_t* coeff);

/* batch_mul — setup-utils/src/helpers.rs:56-59 (phase2 delta^-1 of the H and L queries,
 * phase2/src/parameters.rs:294-296; phase2/src/chunked_groth16.rs:442-466). */
int ss_batch_mul(int curve, int group, uint8_t* bases, size_t n, const uint8_t* coeff);

/* read_batch + write_batch — setup-utils/src/io/read.rs:110-135, io/write.rs:57-66: decode n
 * elements with the given validation and re-encode them (decompress_buffer,
 * phase1/src/helpers/accumulator.rs:182-198, when in_compressed=1,out_compressed=0).
 * out may be NULL to validate only. */
int ss_transcode(int curve, int group, const uint8_t* in, int in_compressed, int check, uint8_t* out,
                 int out_compressed, size_t n);

/* check_subgroup — setup-utils/src/elements.rs:123-150 on n serialized elements. */
int ss_check_subgroup(int curve, int group, const uint8_t* in, int compressed, size_t n, int subgroup_mode);

/* merge_pairs — setup-utils/src/helpers.rs:371-384: (s, sx) = (sum rho_i v1_i, sum rho_i v2_i), both
 * returned as UNCOMPRESSED elements for the caller's check_same_ratio (helpers.rs:410-424; the 2
 * pairings stay on the host).  Randomness: `rho` = n explicit scalars (tests / deterministic callers)
 * or, when NULL, rho_i = first 128 bits of ChaCha20(key = rho_seed[32], counter = i) generated on the
 * device (the reference draws full-width scalars from thread_rng, helpers.rs:373-376; 128 bits keep
 * the soundness error at 2^-128).  Phase 2 uses it for the H and L queries
 * (phase2/src/parameters.rs:393-407, phase2/src/chunked_groth16.rs:521-566). */
int ss_merge_pairs(int curve, int group, const uint8_t* v1, const uint8_t* v2, int compressed, int check, size_t n,
                   const uint8_t* rho, const uint8_t* rho_seed, uint8_t* out_s, uint8_t* out_sx);

/* power_pairs — setup-utils/src/helpers.rs:388-390: merge_pairs(v[..n-1], v[1..]); n-1 scalars. */
int ss_power_pairs(int curve, int group, const uint8_t* v, int compressed, int check, size_t n, const uint8_t* rho,
                   const uint8_t* rho_seed, uint8_t* out_s, uint8_t* out_sx);

/* -------------------------------------------------------------------------------------------- */
/* phase1 helpers                                                                               */
/* -------------------------------------------------------------------------------------------- */
/* check_elements_are_nonzero_and_in_prime_order_subgroup + check_power_ratios(_g2) + re-emit —
 * phase1/src/helpers/accumulator.rs:95-145,56-91 and the write_batch of
 * phase1/src/verification.rs:271-274, fused over ONE decode of the n elements:
 *   - decode with CheckForCorrectness::OnlyNonZero (infinity => SS_ERR_POINT_AT_INFINITY)
 *   - unless subgroup_mode == SS_SUBGROUP_NO: every element must satisfy r*P = O
 *     (else SS_ERR_INCORRECT_SUBGROUP)
 *   - do_ratio: (out_s, out_sx) = power_pairs of the n elements (see ss_merge_pairs for rho)
 *   - out != NULL: the elements re-encoded with out_compressed. */
int ss_check_and_ratio(int curve, int group, const uint8_t* in, int in_compressed, size_t n, int subgroup_mode,
                       int do_ratio, const uint8_t* rho, const uint8_t* rho_seed, uint8_t* out, int out_compressed,
                       uint8_t* out_s, uint8_t* out_sx);

/* apply_powers — phase1/src/helpers/buffers.rs:77-97, fused with generate_powers_of_tau.
 * in/out point at element `start` of the vector (the caller has applied start*size already);
 * n = end - start.  Scalars: `powers` (n explicit scalars) when non-NULL, otherwise
 * tau^(first_power + i).  `coeff` NULL or one scalar (alpha / beta). */
int ss_apply_powers(int curve, int group, const uint8_t* in, int in_compressed, int in_check, uint8_t* out,
                    int out_compressed, size_t n, const uint8_t* powers, const uint8_t* tau, uint64_t first_power,
                    const uint8_t* coeff);

/* Phase1Parameters — phase1/src/objects/parameters.rs:115-294 */
typedef struct {
    int curve;             /* ss_curve */
    int proving_system;    /* ss_proving_system */
    int contribution_mode; /* ss_contribution_mode */
    uint64_t chunk_index;
    uint64_t chunk_size;
    uint32_t total_size_in_log2;
    uint64_t batch_size;
} ss_phase1_params;

typedef struct {
    uint64_t powers_length, powers_g1_length, g1_chunk_size, other_chunk_size;
    uint64_t accumulator_size, contribution_size, public_key_size, hash_size;
} ss_phase1_sizes;

int ss_phase1_sizes_of(const ss_phase1_params* p, ss_phase1_sizes* out);

/* Phase1::initialization — phase1/src/initialization.rs:12-57: the blank accumulator (every element = the group
 * generator, BatchSerializer::init_element, setup-utils/src/io/write.rs:45-55).  The hash prefix is not written. */
int ss_phase1_initialization(const ss_phase1_params* p, uint8_t* output, size_t output_len, int compressed_output);

/* iter_chunk — phase1/src/helpers/buffers.rs:22-73: the window schedule (start, end) of the reference's
 * batch loop (windows overlap by one element).  starts/ends may be NULL to query *count only. */
int ss_phase1_iter_chunk(const ss_phase1_params* p, uint64_t* starts, uint64_t* ends, size_t max_windows, size_t* count);

/* Phase1::computation — phase1/src/computation.rs:16-308 (Groth16 branch :40-193).
 * input/output are the whole challenge / response buffers including the 64-byte hash prefix
 * (which is not touched, as in the reference); tau/alpha/beta = PrivateKey scalars. */
int ss_phase1_computation(const ss_phase1_params* p, const uint8_t* input, size_t input_len, uint8_t* output,
                          size_t output_len, int compressed_input, int compressed_output, int check_input,
                          const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta);

/* Same computation on buffers that already live in device memory of the current device
 * (bench: throughput with inputs resident in HBM).  `stream` is a cudaStream_t. */
int ss_phase1_computation_dev(const ss_phase1_params* p, const void* d_input, size_t input_len, void* d_output,
                              size_t output_len, int compressed_input, int compressed_output, int check_input,
                              const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta, void* stream);

/* Index-range shards of ONE ceremony (SURVEY.md §8e; the chunk ranges of phase1/src/objects/parameters.rs:248-294 cut
 * finer): every vector of the buffer described by `p` is divided into `shard_count` equal contiguous parts and the
 * call processes part `shard_index`; element i of a vector still receives tau^(first + i).  `input` / `output` are
 * the WHOLE challenge / response buffers (typically the same files mapped by one process per GPU) and only the
 * shard's byte ranges are read and written — the contract the reference's sibling rayon tasks already rely on
 * (computation.rs:82-186).  beta_g2 belongs to shard 0.  No inter-process traffic.  With several devices selected in
 * ss_init the shard is divided once more among them. */
int ss_phase1_computation_shard(const ss_phase1_params* p, const uint8_t* input, size_t input_len, uint8_t* output,
                                size_t output_len, int compressed_input, int compressed_output, int check_input,
                                const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta, uint32_t shard_index,
                                uint32_t shard_count);
int ss_phase1_computation_shard_dev(const ss_phase1_params* p, const void* d_input, size_t input_len, void* d_output,
                                    size_t output_len, int compressed_input, int compressed_output, int check_input,
                                    const uint8_t* tau, const uint8_t* alpha, const uint8_t* beta, uint32_t shard_index,
                                    uint32_t shard_count, void* stream);

/* The per-vector hot loop of Phase1::verification — phase1/src/verification.rs:217-411 (Groth16) —
 * over a whole response: for tau_g1, tau_g2, alpha_g1, beta_g1: nonzero + subgroup check, the
 * power_pairs (s, sx) for the caller's check_same_ratio, and the vector re-encoded into
 * new_challenge (NULL: aggregate_verification style, no re-emit, verification.rs:505-769);
 * beta_g2 is validated and re-emitted too (verification.rs:199-201).
 * `pairs`: 4 x (s || sx), uncompressed, in the order tau_g1, tau_g2, alpha_g1, beta_g1
 * (2*g1, 2*g2, 2*g1, 2*g1 uncompressed sizes).  The O(1) proof-of-knowledge / generator /
 * before-after pairing checks on the first elements (verification.rs:83-213) and the 8 pairings on
 * `pairs` stay with the caller.  The 64-byte hash prefix of new_challenge is not written. */
int ss_phase1_verification_vectors(const ss_phase1_params* p, const uint8_t* output, size_t output_len,
                                   int compressed_output, uint8_t* new_challenge, size_t new_challenge_len,
                                   int compressed_new_challenge, int subgroup_mode, int ratio_check,
                                   const uint8_t* rho_seed, uint8_t* pairs);

/* Accumulator re-layout (SURVEY.md §8f rank 1) — read_batch(CheckForCorrectness::No) -> write_batch streams:
 *   ss_phase1_aggregate_chunk — one iteration of Phase1::aggregation (phase1/src/aggregation.rs:11-180): the
 *     vectors of chunk `chunk_params->chunk_index` are written into the full accumulator at
 *     chunk_index*chunk_size (beta_g2 comes from chunk 0);
 *   ss_phase1_split_chunk — one iteration of Phase1::split (aggregation.rs:189-353), the reverse;
 *   ss_phase1_decompress — helpers::accumulator::decompress (accumulator.rs:200-301): compressed
 *     accumulator -> uncompressed, elements read with `check`.
 * `chunk_params` must be in SS_MODE_CHUNKED; `full` is laid out for the same power in full mode.  The
 * 64-byte hash prefixes are not touched. */
int ss_phase1_aggregate_chunk(const ss_phase1_params* chunk_params, const uint8_t* chunk, size_t chunk_len, int compressed_chunk,
                              uint8_t* full, size_t full_len, int compressed_full);
int ss_phase1_split_chunk(const ss_phase1_params* chunk_params, const uint8_t* full, size_t full_len, int compressed_full,
                          uint8_t* chunk, size_t chunk_len, int compressed_chunk);
int ss_phase1_decompress(const ss_phase1_params* p, const uint8_t* in, size_t in_len, int check, uint8_t* out, size_t out_len);

/* Same on buffers resident in device memory (`pairs` and rho_seed stay host pointers). */
int ss_phase1_verification_vectors_dev(const ss_phase1_params* p, const void* d_output, size_t output_len,
                                       int compressed_output, void* d_new_challenge, size_t new_challenge_len,
                                       int compressed_new_challenge, int subgroup_mode, int ratio_check,
                                       const uint8_t* rho_seed, uint8_t* pairs, void* stream);

/* Shard `shard_index` of `shard_count` of the verification loop (see ss_phase1_computation_shard).  The shard reads
 * ONE element beyond its range where its last ratio pair continues into the next shard (power_pairs pairs v[i] with
 * v[i+1], setup-utils/src/helpers.rs:388-390 — the reason iter_chunk overlaps its windows, buffers.rs:54); rho_i is
 * keyed by the global element index.  `pairs` receives the shard's PARTIAL sums (an empty shard: identities). */
int ss_phase1_verification_vectors_shard(const ss_phase1_params* p, const uint8_t* output, size_t output_len,
                                         int compressed_output, uint8_t* new_challenge, size_t new_challenge_len,
                                         int compressed_new_challenge, int subgroup_mode, int ratio_check,
                                         const uint8_t* rho_seed, uint8_t* pairs, uint32_t shard_index, uint32_t shard_count);
int ss_phase1_verification_vectors_shard_dev(const ss_phase1_params* p, const void* d_output, size_t output_len,
                                             int compressed_output, void* d_new_challenge, size_t new_challenge_len,
                                             int compressed_new_challenge, int subgroup_mode, int ratio_check,
                                             const uint8_t* rho_seed, uint8_t* pairs, uint32_t shard_index,
                                             uint32_t shard_count, void* stream);

/* Bytes of a `pairs` blob (2 * (3 * g1_uncompressed + g2_uncompressed)), and the host-side reduction of SURVEY.md §8e:
 * pairs <- element-wise group sums of `count` partial blobs laid out back to back.  The sum of the shards' partial
 * (s, sx) is itself a valid random linear combination, so the caller's check_same_ratio runs on it unchanged. */
size_t ss_phase1_pairs_size(int curve);
int ss_phase1_reduce_partial_pairs(int curve, const uint8_t* partials, int count, uint8_t* pairs);

/* -------------------------------------------------------------------------------------------- */
/* prepare_phase2: powers of tau -> Lagrange coefficients (SURVEY.md §8f rank 3)                */
/* -------------------------------------------------------------------------------------------- */
/* to_coeffs — setup-utils/src/groth16_utils.rs:44-53: `domain.ifft` over the group followed by
 * normalize_batch, on n serialized elements (n a power of two, the radix-2 domain of that size):
 *   out_j = (1/n) * sum_i w^(-i*j) * in_i,   w = Fr::get_root_of_unity(n)
 * (ark-ff 0.4: TWO_ADIC_ROOT_OF_UNITY = GENERATOR^((r-1)/2^s) squared down to order n). */
int ss_group_ifft(int curve, int group, const uint8_t* in, int in_compressed, int check, size_t n, uint8_t* out,
                  int out_compressed);

/* h_query_groth16 — setup-utils/src/groth16_utils.rs:59-63: out_i = powers[i + degree] - powers[i] for
 * i < degree - 1 (G1).  n_powers < 2*degree - 1 => SS_ERR_INVALID_LENGTH (the reference panics). */
int ss_h_query_groth16(int curve, const uint8_t* powers, int in_compressed, int check, size_t n_powers, size_t degree,
                       uint8_t* out, int out_compressed);

/* domain_size (groth16_utils.rs:65-69) and the byte length Groth16Params::write produces
 * (groth16_utils.rs:134-168): alpha_g1, beta_g1, beta_g2, coeffs_g1[m], coeffs_g2[m],
 * alpha_coeffs_g1[m], beta_coeffs_g1[m], h_g1[m-1].  m above 2^(2-adicity of Fr) has no radix-2 domain =>
 * SS_ERR_INVALID_ARGUMENT (only MNT6-753, 2-adicity 15, reaches that at practical sizes). */
int ss_groth16_params_size(int curve, uint64_t phase2_size, int compressed, uint64_t* domain_size, size_t* bytes);

/* Groth16Params::new + ::write — setup-utils/src/groth16_utils.rs:81-131,134-168, the body of
 * prepare_phase2 (phase2-cli/src/prepare_phase2.rs:16-70): `accumulator` is a full-mode Groth16 phase-1
 * accumulator (64-byte hash prefix included, as Phase1::deserialize takes it); elements are read with
 * `check`.  A domain larger than the accumulator's powers => SS_ERR_INVALID_LENGTH (reference: slice panic). */
int ss_groth16_params_new(const ss_phase1_params* p, const uint8_t* accumulator, size_t accumulator_len,
                          int compressed_input, int check, uint64_t phase2_size, uint8_t* out, size_t out_len,
                          int compressed_output);

/* -------------------------------------------------------------------------------------------- */
/* ratio checks by pairing (SURVEY.md §8 A12, §8f rank 2)                                       */
/* -------------------------------------------------------------------------------------------- */
/* same_ratio — setup-utils/src/helpers.rs:406-408: *same = (e(g1.0, g2.1) == e(g1.1, g2.0)).
 * g1_pair = g1.0 || g1.1 and g2_pair = g2.0 || g2.1, UNCOMPRESSED elements (what ss_power_pairs /
 * ss_merge_pairs / ss_phase1_verification_vectors return).  The device evaluates a reduced Tate pairing
 * product; the verdict is the same for every non-degenerate pairing on G1 x G2.  Inputs must be subgroup
 * points (the callers have checked that), e(O, .) = 1. */
int ss_same_ratio(int curve, const uint8_t* g1_pair, const uint8_t* g2_pair, int* same);

/* check_same_ratio — setup-utils/src/helpers.rs:410-424: SS_ERR_INVALID_RATIO when one of the four points
 * is zero or the pairings differ. */
int ss_check_same_ratio(int curve, const uint8_t* g1_pair, const uint8_t* g2_pair);

/* `count` independent checks in one launch (one warp each), e.g. the four vectors of a response;
 * *first_bad = index of the first failing check. */
int ss_check_same_ratio_batch(int curve, const uint8_t* g1_pairs, const uint8_t* g2_pairs, int count, int* first_bad);

/* The per-vector half of Phase1::verification WITH its verdict (phase1/src/verification.rs:44-80,217-411):
 * ss_phase1_verification_vectors followed by check_power_ratios / check_power_ratios_g2 for every vector
 * (phase1/src/helpers/accumulator.rs:56-91) against g2_check = (tau_g2[0], tau_g2[1]) and
 * g1_check = (tau_g1[0], tau_g1[1]) read from the response with `check_output` (verification.rs:58-71).
 * SS_ERR_INVALID_RATIO: ss_last_error().index = 0 tau_g1, 1 tau_g2, 2 alpha_g1, 3 beta_g1.  The proof-of-knowledge
 * and before/after checks on the first elements (verification.rs:83-213) need hash_to_g2 and stay with the
 * caller, who can run their check_same_ratio through ss_check_same_ratio_batch. */
int ss_phase1_verification_ratios(const ss_phase1_params* p, const uint8_t* output, size_t output_len, int compressed_output,
                                  int check_output, uint8_t* new_challenge, size_t new_challenge_len,
                                  int compressed_new_challenge, int subgroup_mode, const uint8_t* rho_seed);

/* check_power_ratios / check_power_ratios_g2 (phase1/src/helpers/accumulator.rs:56-91) of the four vectors from their
 * (s, sx) `pairs` — whole-response pairs or the ss_phase1_reduce_partial_pairs of the shards' blobs — and
 * g1_check = tau_g1[0] || tau_g1[1], g2_check = tau_g2[0] || tau_g2[1] (uncompressed, verification.rs:58-71).
 * SS_ERR_INVALID_RATIO: ss_last_error().index = failing vector. */
int ss_phase1_check_ratio_pairs(int curve, const uint8_t* pairs, const uint8_t* g1_check, const uint8_t* g2_check);

/* -------------------------------------------------------------------------------------------- */
/* phase-2 QAP evaluation (SURVEY.md §8f rank 4)                                                */
/* -------------------------------------------------------------------------------------------- */
/* dot_product_vec + normalize_batch — phase2/src/polynomial.rs:30-47,75-94:
 *   out_v = sum_{e in [row_ptr[v], row_ptr[v+1])} coeffs[e] * bases[index[e]],   v < rows
 * `bases`: n_bases serialized elements (the Lagrange coefficients of Groth16Params); the matrix is the
 * per-variable list `xt_processed` of MPCParameters::process_matrix (phase2/src/parameters.rs:96-105) in CSR
 * form: row_ptr[rows + 1], index[nnz] (constraint numbers), coeffs[nnz] canonical little-endian scalars.
 * A row without entries gives the point at infinity, as the reference's empty sum does.  dot_product_ext
 * (polynomial.rs:51-68) is the same call over the concatenation [beta_coeffs | alpha_coeffs | coeffs_g1] with
 * the indices of bt / ct shifted by m / 2m.  An index >= n_bases => SS_ERR_INVALID_LENGTH (reference: panic). */
int ss_qap_dot_product(int curve, int group, const uint8_t* bases, int bases_compressed, int check, size_t n_bases,
                       const uint64_t* row_ptr, const uint32_t* index, const uint8_t* coeffs, size_t rows, uint8_t* out,
                       int out_compressed);

#ifdef __cplusplus
}
#endif
#endif /* SNARK_SETUP_B200_H */
