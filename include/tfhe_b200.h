/*
 * tfhe_b200.h -- C ABI of the B200-native KS-PBS engine (libtfhe_b200.so, CUDA sm_100a).
 *
 * The reference (tfhe-rs 0.5.0 fork, /root/reference) has NO FFI under this path: KS-PBS is a direct
 * Rust call chain (SURVEY.md section 3.2).  This boundary is introduced exactly under
 *   shortint::ServerKey::apply_lookup_table        tfhe/src/shortint/server_key/mod.rs:457-476
 *   ServerKey::keyswitch_programmable_bootstrap_assign                         mod.rs:783-857
 * and follows the reference's own C-API conventions (tfhe/src/c_api/utils.rs:3-28): every function
 * returns int, 0 = success, non-zero = failure; out-pointers are nulled first; objects are opaque
 * heap handles freed by a matching destroy; raw key / ciphertext arrays stay caller-owned
 * (precedent: tfhe/src/c_api/core_crypto/mod.rs:38-122).  INTEGRATION.md shows the Rust
 * `extern "C"` block and build.rs lines a maintainer would add.
 *
 * Only raw LWE arrays cross the boundary; degree / noise-level metadata and the trivial-ciphertext
 * short cut (mod.rs:788-791) stay on the host side.
 */
#ifndef TFHE_B200_H
#define TFHE_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tfhe_b200_ctx tfhe_b200_ctx;

/* shortint::ClassicPBSParameters / MultiBitPBSParameters (shortint/parameters/mod.rs:598-1136,
 * multi_bit.rs:96-209); grouping_factor = 0 selects the classic PBS, 2 or 3 the multi-bit PBS.
 * Accepted: every PARAM_MESSAGE_m_CARRY_c_KS_PBS (N = 256 ... 32768, k = 1 ... 5, 1 ... 3 PBS levels) and
 * every PARAM_MULTI_BIT_MESSAGE_m_CARRY_c_GROUP_g_KS_PBS (N <= 8192).  N = 2048, k = 1, one PBS level
 * (classic, and multi-bit with g = 3) runs on the tuned kernels, everything else on the generic one. */
typedef struct {
    uint32_t lwe_dim;        /* n   (small key)            */
    uint32_t glwe_dim;       /* k                           */
    uint32_t poly_size;      /* N                           */
    uint32_t pbs_base_log, pbs_level;
    uint32_t ks_base_log, ks_level;
    uint32_t grouping_factor;
    uint32_t msg_mod, carry_mod;
} tfhe_b200_params;

/* Lifetime.  One context per GPU; re-entrant per context, no thread-locals (replaces the thread-local
 * ShortintEngine scratch, shortint/engine/mod.rs:23-25,184-189, and the global FFT plan cache,
 * core_crypto/fft_impl/fft64/math/fft/mod.rs:98-102,146-193). */
int tfhe_b200_ctx_create(int cuda_device, const tfhe_b200_params *params, tfhe_b200_ctx **out);
int tfhe_b200_ctx_destroy(tfhe_b200_ctx *ctx);
const char *tfhe_b200_last_error(void);
/* CiphertextModulus (core_crypto/commons/ciphertext_modulus.rs): native 2^64 by default; a smaller power of two 2^log2_q keeps its
 * values in the MSBs of each u64 word and makes every PBS output round to a multiple of 2^(64 - log2_q), exactly as
 * fft64/crypto/bootstrap.rs:318-330 does.  The keyswitch is unchanged (lwe_keyswitch.rs:136-140: compatible with the native modulus). */
int tfhe_b200_set_ciphertext_modulus_log2(tfhe_b200_ctx *ctx, uint32_t log2_q);

/* Keys (host pointers, copied).
 * ksk: LweKeyswitchKey<u64> container, [k*N][ks_level (level l..1)][n+1]
 *      (core_crypto/entities/lwe_keyswitch_key.rs:77-110,396).
 * bsk: STANDARD-domain LweBootstrapKey<u64>, [n][pbs_level (1..l)][k+1][k+1][N]
 *      (entities/ggsw_ciphertext.rs:185-197); converted to the engine's own Fourier layout on the
 *      device (replaces lwe_bootstrap_key_conversion.rs:99- / FourierLweBootstrapKey::new).
 * luts: n_luts accumulators as produced by ServerKey::generate_lookup_table
 *      (shortint/server_key/mod.rs:383-399, engine/mod.rs:72-128), each (k+1)*N words. */
int tfhe_b200_upload_ksk(tfhe_b200_ctx *ctx, const uint64_t *ksk, size_t len);
int tfhe_b200_upload_bsk_std(tfhe_b200_ctx *ctx, const uint64_t *bsk, size_t len);
int tfhe_b200_upload_luts(tfhe_b200_ctx *ctx, const uint64_t *luts, uint32_t n_luts);

/* Seeded (compressed) keys: what shortint::CompressedServerKey holds (shortint/server_key/mod.rs:935-1023) -- per key a 128-bit
 * compression seed and the ciphertext BODIES only.  Replaces SeededLweKeyswitchKey::par_decompress_into_lwe_keyswitch_key
 * (core_crypto/algorithms/seeded_lwe_keyswitch_key_decompression.rs, seeded_lwe_ciphertext_list_decompression.rs:9-60) and
 * SeededLweBootstrapKey / SeededLweMultiBitBootstrapKey::par_decompress_into_* followed by the Fourier conversion
 * (seeded_lwe_bootstrap_key_decompression.rs, seeded_ggsw_ciphertext_list_decompression.rs, seeded_glwe_ciphertext_decompression.rs):
 * the masks are re-drawn ON THE DEVICE from concrete-csprng's AES-128 CTR stream (bit-exact with the reference's generator).
 * seed:   the 16 bytes of Seed(u128).0.to_ne_bytes() (little endian), i.e. the AES key of soft/block_cipher.rs:16.
 * bodies: ksk: [k*N][ks_level] one word per LWE ciphertext (entities/seeded_lwe_keyswitch_key.rs);
 *         bsk: [n or groups*2^g][pbs_level][k+1 rows][N] one body polynomial per GLWE row (entities/seeded_ggsw_ciphertext_list.rs). */
int tfhe_b200_upload_seeded_ksk(tfhe_b200_ctx *ctx, const uint8_t seed[16], const uint64_t *bodies, size_t len);
int tfhe_b200_upload_seeded_bsk(tfhe_b200_ctx *ctx, const uint8_t seed[16], const uint64_t *bodies, size_t len);

/* tfhe-rs wire format (SURVEY 8(f) N3): bincode 1.3.3 with fixed-width little-endian integers, i.e. what `bincode::serialize` and
 * safe_serialize (tfhe/src/safe_deserialization.rs:13-34) emit, for shortint::CompressedServerKey (shortint/server_key/compressed.rs:
 * 10-17,43-55), shortint::Ciphertext (shortint/ciphertext/mod.rs:261-270) and BaseRadixCiphertext { blocks: Vec<Ciphertext> }
 * (integer/ciphertext/mod.rs:18-30).  Layout restated from the serde derives (fhe_string_bounty_b200/csrc/host/wire.h); no real
 * tfhe-rs blob is available in this environment to pin it ("parity unpinned").
 * parse_compressed_server_key: no GPU needed; tells the caller which parameter set to create the context with.
 * load_compressed_server_key:  parse + tfhe_b200_upload_seeded_ksk + tfhe_b200_upload_seeded_bsk.
 * read/write_ciphertexts:      lwe = n_cts x lwe_len words; meta = 5 words per ciphertext {degree, noise_level, message_modulus,
 *                              carry_modulus, pbs_order}.  Pass lwe_out / out = NULL to query the sizes. */
typedef struct {
    tfhe_b200_params params;
    uint32_t pbs_order;                 /* core_crypto/commons/parameters.rs:233-245: 0 = KeyswitchBootstrap, 1 = BootstrapKeyswitch */
    uint32_t deterministic_execution;   /* multi-bit only */
    uint64_t max_degree;
    uint8_t ksk_seed[16], bsk_seed[16];
    uint64_t ksk_byte_offset, ksk_words, bsk_byte_offset, bsk_words;   /* where the two body arrays sit inside the blob */
} tfhe_b200_wire_server_key;
int tfhe_b200_wire_parse_compressed_server_key(const uint8_t *bytes, size_t len, tfhe_b200_wire_server_key *out);
int tfhe_b200_load_compressed_server_key(tfhe_b200_ctx *ctx, const uint8_t *bytes, size_t len);
int tfhe_b200_wire_read_ciphertexts(const uint8_t *bytes, size_t len, int is_radix, uint64_t *lwe_out, size_t lwe_cap_words,
                                    uint64_t *meta_out, size_t *n_cts, size_t *lwe_len);
int tfhe_b200_wire_write_ciphertexts(const uint64_t *lwe, size_t lwe_len, const uint64_t *meta, size_t n_cts, int is_radix,
                                     uint8_t *out, size_t out_cap, size_t *out_len);

/* Batched hot path, HOST buffers (H2D + kernels + D2H inside the call, synchronous).
 * lwe_big:   batch x (k*N + 1) words under the big key;  lwe_small: batch x (n + 1) words.
 * lut_idx:   batch indices into the uploaded LUT table (NULL = LUT 0 for all).
 * keyswitch_batch  replaces keyswitch_lwe_ciphertext            core_crypto/algorithms/lwe_keyswitch.rs:96-170
 * pbs_batch        replaces programmable_bootstrap_lwe_ciphertext_mem_optimized
 *                                                                algorithms/lwe_programmable_bootstrapping.rs:1067-1107
 * ks_pbs_batch     replaces keyswitch_programmable_bootstrap_assign (non-trivial branch)
 *                                                                shortint/server_key/mod.rs:793-856 */
int tfhe_b200_keyswitch_batch(tfhe_b200_ctx *ctx, const uint64_t *lwe_big, uint64_t *lwe_small, size_t batch);
int tfhe_b200_pbs_batch(tfhe_b200_ctx *ctx, const uint64_t *lwe_small, const uint32_t *lut_idx, uint64_t *lwe_big,
                        size_t batch);
int tfhe_b200_ks_pbs_batch(tfhe_b200_ctx *ctx, const uint64_t *lwe_big_in, const uint32_t *lut_idx,
                           uint64_t *lwe_big_out, size_t batch);
/* PBS -> KS order (PBSOrder::BootstrapKeyswitch; programmable_bootstrap_keyswitch_assign, shortint/server_key/mod.rs:859-932):
 * ciphertexts are batch x (n + 1) words under the SMALL key on both sides. */
int tfhe_b200_pbs_ks_batch(tfhe_b200_ctx *ctx, const uint64_t *lwe_small_in, const uint32_t *lut_idx,
                           uint64_t *lwe_small_out, size_t batch);

/* Same operations on DEVICE buffers of the context's GPU, enqueued on `cuda_stream` (a cudaStream_t;
 * NULL = the context's own stream) without synchronising: used to chain tree levels and by the
 * multi-GPU driver. */
int tfhe_b200_keyswitch_batch_device(tfhe_b200_ctx *ctx, const uint64_t *d_lwe_big, uint64_t *d_lwe_small, size_t batch,
                                     void *cuda_stream);
int tfhe_b200_pbs_batch_device(tfhe_b200_ctx *ctx, const uint64_t *d_lwe_small, const uint32_t *d_lut_idx,
                               uint64_t *d_lwe_big, size_t batch, void *cuda_stream);
int tfhe_b200_ks_pbs_batch_device(tfhe_b200_ctx *ctx, const uint64_t *d_lwe_big_in, const uint32_t *d_lut_idx,
                                  uint64_t *d_lwe_big_out, size_t batch, void *cuda_stream);
int tfhe_b200_synchronize(tfhe_b200_ctx *ctx);

/* Test hook: PBS that stops after `n_iters` blind-rotation iterations (n_iters = 1 gives one CMUX =
 * one add_external_product_assign, fft64/crypto/ggsw.rs:477-598, whose output is comparable
 * coefficient-wise with the oracle). */
int tfhe_b200_pbs_batch_partial(tfhe_b200_ctx *ctx, const uint64_t *lwe_small, const uint32_t *lut_idx,
                                uint64_t *lwe_big, size_t batch, uint32_t n_iters);

/* ---- host layer: integer-radix / string operations recorded as level-batched programs -------------------------
 * Mirrors, as one batched call per tree level, the per-block rayon fan-out of
 *   integer::ServerKey::{unchecked_eq,ne,lt,le,gt,ge}_parallelized   integer/server_key/radix_parallel/comparison.rs:10-83,
 *                                                                      integer/server_key/comparator.rs:389-464,1103-1126
 *   are_all_comparisons_block_true / is_at_least_one_...              radix_parallel/scalar_comparison.rs:147-240
 *   unchecked_scalar_{eq,lt,gt}_parallelized                          scalar_comparison.rs:366-458, comparator.rs:474-502
 *   if_then_else_parallelized                                         radix_parallel/cmux.rs:72-
 *   add_parallelized (carry propagation)                              radix_parallel/add.rs:206-243,518-603
 * and the string compositions of SURVEY.md Appendix B (the snapshot has no FheString module; see
 * fhe_string_bounty_b200/csrc/host/strings.h).  `op` is one of:
 *   shortint_apply_lut {n, f(0..15)}      shortint_bivariate_lut {n, f(x,y) row-major}
 *   radix_{eq,ne,lt,le,gt,ge,add} {n_blocks}   radix_scalar_{eq,lt,gt} {n_blocks, scalar}   radix_if_then_else {n_blocks}
 *   radix_default_{eq,ne,lt,le,gt,ge} {n_blocks, block_degree} / radix_full_propagate {n_blocks, block_degree}: operands whose carries
 *     are not empty (degree up to msg_mod*carry_mod - 1) are propagated first, as the non-"unchecked" reference methods do
 *   bool_all_true / bool_any_true {n}     bool_sum_finish {n_summed, want_all}
 *   string_{eq,ne,lt,le,gt,ge,eq_ignore_case,contains,starts_with,ends_with,find} {len_a, len_b}
 *   string_{to_lowercase,to_uppercase} {len}     string_contains_windows {len_a, len_b, w0, w1}
 *   string_{eq,ne,lt,le,contains}_many {len_a, len_b, count}   (count independent pairs in one program)
 *   pstring_{len,is_empty,trim_start,trim_end,trim} {capacity}     pstring_{strip_prefix,strip_suffix} {capacity} + clear pattern
 *   pstring_{eq,ne,lt,le,gt,ge,contains,starts_with,ends_with,find,rfind,concat} {capacity_a, capacity_b}     pstring_repeat {capacity, count}
 *   pstring_replace {capacity, capacity_from, capacity_to}  pstring_replacen {capacity, capacity_from, capacity_to, count}: inputs s, from,
 *     to -> C = capacity + min(count, M) * max(0, capacity_to - m_min) chars (replace: count unbounded)
 *   pstring_split {capacity, capacity_pat}  pstring_splitn {capacity, capacity_pat, n}: inputs s, pat -> the part count (ceil(log4(P + 1))
 *     blocks), then P parts of capacity chars, P = M + 1 (splitn: min(M + 1, n); the last part is the unsplit rest; n = 0: count 0)
 *   pstring_split_once / pstring_rsplit_once {capacity, capacity_pat}: inputs s, pat -> found, before, after (capacity chars each; both
 *     empty when nothing is found).  rsplit_once splits at the last match as rfind finds it
 *   pstring_{rsplit,split_terminator,rsplit_terminator,split_inclusive} {capacity, capacity_pat}  pstring_rsplitn {capacity, capacity_pat, n}:
 *     inputs s, pat -> the part count (ceil(log4(P + 1)) blocks), then P parts of capacity chars, P = M + 1 (rsplitn: min(M + 1, n)).
 *     rsplit / rsplitn: the rightmost non-overlapping matches, parts in Rust's order from the end (rsplitn: the last part is the unsplit
 *     prefix; n = 0: count 0).  split_terminator / rsplit_terminator: split / rsplit without the part at the end of the string when that
 *     part is empty.  split_inclusive: each part keeps the match that ends it; an empty part at the end is dropped
 *   pstring_split_ascii_whitespace {capacity}: input s -> the word count, then P = ceil(capacity / 2) words of capacity chars; words are
 *     separated by the bytes of u8::is_ascii_whitespace (U+0009, U+000A, U+000C, U+000D, U+0020; not U+000B)
 *   secret integers (the _enc ops): a radix of count_blocks 2-bit blocks (1 ..= 16, little endian), the last input
 *   pstring_repeat_enc {capacity, max_count, count_blocks}: inputs s, count -> capacity * max_count chars: s repeated min(count, max_count)
 *     times (a count above max_count is clamped to it)
 *   pstring_replacen_enc {capacity, capacity_from, capacity_to, count_blocks}: inputs s, from, to, count -> the first `count` matches
 *     replaced (all of them when count >= M), in the C = capacity + M * max(0, capacity_to - m_min) chars of replace
 *   pstring_splitn_enc / pstring_rsplitn_enc {capacity, capacity_pat, n_blocks}: inputs s, pat, n -> the part count (ceil(log4(M + 2))
 *     blocks), then M + 1 parts of capacity chars: splitn / rsplitn with n parts at most (n = 0: count 0)
 *   pstring_{strip_prefix,strip_suffix} {capacity, capacity_pat} without a clear operand: inputs s, pat (padded) -> matched, the string
 *   pstring_eq_ignore_case {capacity_a, capacity_b}: inputs a, b (or a and the clear b, capacity_b its length) -> one boolean block:
 *     a and b equal after the ASCII case fold
 *   pstring_matches {capacity, capacity_pat}: inputs s, pat -> s.matches(pat).count() as ceil(log4(M + 1)) blocks.  There is no separate
 *     rmatches count: with every match of one length, greedy selection from the left and from the right both find a largest set of
 *     non-overlapping matches, so the two counts are equal (the empty pattern: len + 1 either way)
 *   pstring_match_indices / pstring_rmatch_indices {capacity, capacity_pat}: inputs s, pat -> the count (ceil(log4(M + 1)) blocks), then
 *     M byte indices of ceil(log4(capacity + 1)) blocks each: the leftmost non-overlapping matches in order (rmatch_indices: the
 *     rightmost ones as the reverse searcher finds them, last match first); indices past the count are zero.  M * (capacity + 1) is
 *     limited to 2^20
 *   pstring_trim_start_matches / pstring_trim_end_matches {capacity, capacity_pat}: inputs s, pat -> capacity chars: s without the run of
 *     back-to-back matches at its start / at its (secret) end; the empty pattern returns s
 *   pstring_lines {capacity}: input s -> the line count (ceil(log4(capacity + 1)) blocks), then capacity lines of capacity chars: s split
 *     after every "\n", each line without its "\n" or "\r\n" (a bare "\r" at the end stays), no empty line after a final "\n"
 *   pstring_split_whitespace {capacity}: input s -> the word count, then P = ceil(capacity / 2) words of capacity chars; words are separated
 *     by char::is_whitespace (Unicode White_Space), i.e. every occurrence of the UTF-8 sequences 09 ..= 0D, 20, C2 85, C2 A0, E1 9A 80,
 *     E2 80 80 ..= E2 80 8A, E2 80 A8, E2 80 A9, E2 80 AF, E2 81 9F, E3 80 80.  For valid UTF-8 that is Rust's result; for other bytes
 *     this rule is the definition.  lines and split_whitespace take no clear operand
 *     -- Rust's str methods with a &str pattern: leftmost non-overlapping matches, the empty pattern matching at every char boundary
 *        0 ..= len.  With clear_operand != NULL it is the pattern (from / pat, not an input) and capacity_from / capacity_pat must equal
 *        its length.  m_min is the least pattern length (0 for a padded pattern, the length of a clear one) and M the most matches:
 *        capacity + 1 when m_min = 0, else capacity / m_min.  Parts past the count are all zero.  Capacities, and the chars of the result
 *        and of replace's expanded string, are limited to 2^20.
 *     -- NULL-PADDED strings: public capacity, secret length, content followed by zero bytes (host/padded.h); len returns a radix of
 *        ceil(log4(capacity + 1)) blocks, the string-valued ops return 4 blocks per char of the result capacity
 * Appending "_packed" to a string op (or radix_eq) selects packed block equalities: one PBS per PAIR of blocks built from
 * pack_block_chunk + lwe_sub + LUT[x == 0] (the Comparator's own trick, comparator.rs:193-221); same decrypted results.
 * With clear_operand != NULL the second string operand is that clear (trivial) string instead of an input.
 * Inputs are fresh shortint blocks (degree msg_mod-1); a char is ceil(8 / log2(msg_mod)) little-endian blocks (4 two-bit blocks for the
 * MESSAGE_2 sets).  to_lowercase / to_uppercase / eq_ignore_case / find and the pstring_* operations require msg_mod = 4. */
typedef struct tfhe_b200_program tfhe_b200_program;
int tfhe_b200_program_build(const tfhe_b200_params *params, const char *op, const uint64_t *args, size_t n_args,
                            const char *clear_operand, tfhe_b200_program **out);
int tfhe_b200_program_destroy(tfhe_b200_program *prog);
int tfhe_b200_program_counts(const tfhe_b200_program *prog, uint64_t counts[9]);
int tfhe_b200_program_copy(const tfhe_b200_program *prog, uint32_t *level_lin_off, uint32_t *level_pbs_off,
                           uint32_t *lin_out_tb_te, uint64_t *lin_body, uint32_t *term_slot, int64_t *term_coef,
                           uint32_t *pbs_in_out_lut, uint64_t *lut_tables, uint64_t *lut_degrees, uint32_t *outputs,
                           uint64_t *output_degree_noise);
int tfhe_b200_program_accumulators(const tfhe_b200_program *prog, uint64_t *accs);
int tfhe_b200_program_run(tfhe_b200_ctx *ctx, tfhe_b200_program *prog, const uint64_t *inputs, uint64_t *outputs);
/* Same on DEVICE buffers of the context's GPU, enqueued on `cuda_stream` (NULL = the context's stream) without synchronising; chains a
 * rank's share of a sharded operation, the exchange below and the finishing program with no host round trip in between. */
int tfhe_b200_program_run_device(tfhe_b200_ctx *ctx, tfhe_b200_program *prog, const uint64_t *d_inputs, uint64_t *d_outputs,
                                 void *cuda_stream);
int tfhe_b200_program_last_ms(const tfhe_b200_program *prog, float *ms);

/* ---- multi-GPU: the one exchange step of a sharded string operation, over NVLink peer memory ------------------------------------
 * One process per GPU; keys replicated; haystack windows / chars partitioned (SURVEY.md 8e).  Where the wide levels are sharded, the
 * narrow end of the reduction tree -- which the CPU reference hands over through shared memory inside one rayon reduction
 * (are_all_comparisons_block_true / is_at_least_one_comparisons_block_true, integer/server_key/radix_parallel/scalar_comparison.rs:
 * 147-240; the sign tree, integer/server_key/comparator.rs:257-279,957-971) -- crosses GPUs exactly once.  The engine does that
 * exchange itself: every rank owns a symmetric buffer (CUDA IPC), a rank's last tree level writes its rows straight into its send
 * area, and ONE kernel publishes a flag to every peer, waits for all peers' flags and pulls their rows with peer loads, concatenating
 * (all_gather) or summing them modulo 2^64 = homomorphic addition (all_reduce_sum).  No NCCL call and no host synchronisation sit
 * between a rank's share, the exchange and the finishing program (fhe_string_bounty_b200/csrc/exchange.cu).
 *   create -> handle (64-byte CUDA IPC handle; ship it to every peer by any transport) -> attach (all handles, rank order)
 *   send_rows: where the NEXT exchange's local rows go (max_rows x (k*N+1) words) -- pass it as d_outputs of program_run_device
 *   all_gather: d_out = world parts of gather_stride(rows) words each;  all_reduce_sum: d_out = rows x (k*N+1) words (+1 pad if odd)
 * d_out must be 16-byte aligned.  Destroy the exchange before its context.  attach_local serves several ranks driven by one process
 * (on one GPU use group_run instead of the per-rank calls). */
typedef struct tfhe_b200_exchange tfhe_b200_exchange;
int tfhe_b200_exchange_create(tfhe_b200_ctx *ctx, uint32_t rank, uint32_t world, uint32_t max_rows, tfhe_b200_exchange **out);
int tfhe_b200_exchange_handle(tfhe_b200_exchange *ex, uint8_t handle[64]);
int tfhe_b200_exchange_attach(tfhe_b200_exchange *ex, const uint8_t *handles);
int tfhe_b200_exchange_attach_local(tfhe_b200_exchange *ex, tfhe_b200_exchange *const *peers);
int tfhe_b200_exchange_send_rows(tfhe_b200_exchange *ex, uint64_t **d_rows);
size_t tfhe_b200_exchange_gather_stride(const tfhe_b200_exchange *ex, uint32_t rows);
int tfhe_b200_exchange_all_gather(tfhe_b200_exchange *ex, uint32_t rows, uint64_t *d_out, void *cuda_stream);
int tfhe_b200_exchange_all_reduce_sum(tfhe_b200_exchange *ex, uint32_t rows, uint64_t *d_out, void *cuda_stream);
/* several ranks on ONE GPU (attach_local; the single-GPU tests): all ranks' exchanges as one cooperative launch -- kernels that wait
 * on one another must never be separate launches on one device */
int tfhe_b200_exchange_group_run(tfhe_b200_exchange *const *group, uint32_t world, uint32_t rows, uint64_t *const *d_outs, int reduce,
                                 void *cuda_stream);
int tfhe_b200_exchange_destroy(tfhe_b200_exchange *ex);

/* Running any recorded program across the ranks of an exchange (wide levels split, rows scattered back after each) is declared in
 * tfhe_b200_sharded.h, which includes this header. */

/* Kernel selection (A/B comparisons and the parity tests that pin one kernel instance); the same keys are read from the environment at
 * context creation as TFHE_B200_<KEY>.  Keys: "narrow_kernel" (8 = pbs_v8.cu / pbs_multibit_v8.cu serve levels of at most narrow_max
 * ciphertexts and level tails, 0 = the 1- / 2-ciphertext instances of the wide kernels), "narrow_max" (0 = default: 2 x SM count
 * classic, SM count multi-bit), "ks_kernel" (2 = keyswitch on tcgen05.mma kind::i8 [default], 1 = on mma.sync, 0 = IMAD keyswitch; all three are
 * bit-identical), "narrow_cluster" (1 [default] = levels of at most SM count / 2 ciphertexts put one ciphertext on a two-SM thread-block
 * cluster, pbs_classic_kernel_v8x2 / pbs_multibit_kernel_v8x2; 0 = one SM per ciphertext; identical output words either way),
 * "tuned512_min" (N = 512, k = 3 contexts: batches of at least this many ciphertexts run on pbs_n512.cu, smaller ones on the generic
 * kernel; 0 = default: SM count), "tuned8192" (N = 8192, k = 1, two-level contexts: 1 [default] = pbs_n8192.cu, one ciphertext per two-SM
 * cluster; 0 = generic kernel). */
int tfhe_b200_set_tuning(tfhe_b200_ctx *ctx, const char *key, int value);

/* Instrumentation. */
uint64_t tfhe_b200_kernel_launches(const tfhe_b200_ctx *ctx);   /* kernels launched by this context so far */
int tfhe_b200_time_last_kernels(tfhe_b200_ctx *ctx, float *ks_ms, float *pbs_ms); /* CUDA-event ms of the last ks_pbs call */
int tfhe_b200_probe_fp64_tflops(int cuda_device, double *tflops);  /* dependent-FMA microbenchmark */
const char *tfhe_b200_version(void);
/* How the classic-PBS dispatcher cuts a tree level of `batch` ciphertexts of the headline set into launches on a device with `sms` SMs:
 * counts[0] ciphertexts on the 4-per-SM instance of the wide kernel, then counts[1] on its 3-per-SM instance, then counts[2] on the
 * narrow-level kernels; narrow_max = the widest tail those may take, cluster = two-SM clusters allowed.  Pure host arithmetic. */
void tfhe_b200_plan_classic_level(size_t batch, uint32_t sms, size_t narrow_max, int cluster, size_t counts[3]);

#ifdef __cplusplus
}
#endif
#endif
