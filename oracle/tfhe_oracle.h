/*
 * oracle/tfhe_oracle.h -- CPU restatement of the tfhe-rs 0.5.0 shortint KS-PBS path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the shipped engine: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load it.  The
 * product path (fhe_string_bounty_b200/, include/tfhe_b200.h) never links or calls this code.
 *
 * Parity pinning (SURVEY.md section 8c): the reference is Rust and cannot be built in this image
 * (no cargo/rustc, un-vendored crates), and its FFT lives in the third-party crate
 * concrete-fft = "0.3.0" (tfhe/Cargo.toml:60) whose source is absent.  The reference holds NO
 * ciphertext-level golden vectors for this path; what it pins -- and what tests/test_oracle_kat.py
 * checks this oracle against -- are:
 *   - SignedDecomposer doc KATs (commons/math/decomposition/decomposer.rs:94-95,134-142),
 *   - monomial mul/div doc KATs (algorithms/polynomial_algorithms.rs:305-313),
 *   - FFT roundtrip |d| < 2^14 and product-vs-schoolbook tolerance (fft64/math/fft/tests.rs:44,157-172),
 *   - decrypt-and-compare over all messages (algorithms/test/lwe_keyswitch.rs, lwe_programmable_bootstrapping.rs),
 *   - trivial-PBS == real PBS after decryption (shortint/server_key/tests/shortint.rs:3233-3296),
 *   - the ASCII tutorial KAT (docs/tutorials/ascii_fhe_string.md:140-153),
 *   - seeded keys (csprng_oracle.c): the FIPS-197 AES-128 key schedule and ciphertext held by concrete-csprng's tests
 *     (implem/aesni/block_cipher.rs:188-229, implem/soft/block_cipher.rs:84-113).
 * Integer arithmetic (decomposition, keyswitch, monomial ops, sample extraction, LUT layout) is pinned
 * bit-exactly by those KATs; the f64 FFT result bits are "parity unpinned" (tolerance pins only), so
 * an EXACT integer external product (no FFT) is provided as independent ground truth.
 */
#ifndef TFHE_ORACLE_H
#define TFHE_ORACLE_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* shortint/parameters/mod.rs:703-717 (classic), multi_bit.rs:173-190 (multi-bit, grouping_factor=3) */
typedef struct {
    uint32_t lwe_dim;         /* n */
    uint32_t glwe_dim;        /* k */
    uint32_t poly_size;       /* N */
    uint32_t pbs_base_log, pbs_level;
    uint32_t ks_base_log, ks_level;
    uint32_t grouping_factor; /* 0 = classic PBS */
    uint32_t msg_mod, carry_mod;
    double lwe_std, glwe_std;
} orc_params;

void orc_params_message_2_carry_2_ks_pbs(orc_params *p);
void orc_params_multi_bit_message_2_carry_2_group_3_ks_pbs(orc_params *p);
/* small toy set for fast exhaustive tests (not a reference parameter set) */
void orc_params_toy(orc_params *p);

/* seeded PRNG (xoshiro256**, splitmix64 seeding); the Rust AES-CTR stream cannot be reproduced */
typedef struct { uint64_t s[4]; int has_spare; double spare; } orc_rng;
void orc_rng_seed(orc_rng *r, uint64_t seed);
uint64_t orc_rng_u64(orc_rng *r);
double orc_rng_gauss(orc_rng *r);

/* key material ------------------------------------------------------------------------------- */
void orc_gen_binary_key(orc_rng *r, uint64_t *sk, size_t len);
/* lwe_encryption.rs:61-117: ct = (a_0..a_{d-1}, <a,s> + pt + e) */
void orc_lwe_encrypt(const uint64_t *sk, size_t dim, uint64_t plaintext, double std, orc_rng *r, uint64_t *ct);
/* lwe_encryption.rs:520-558 */
uint64_t orc_lwe_decrypt(const uint64_t *sk, size_t dim, const uint64_t *ct);
/* lwe_keyswitch_key_generation.rs:65-131 ; layout [in_dim][level l..1][out_dim+1] */
void orc_gen_ksk(const orc_params *p, const uint64_t *big_sk, const uint64_t *small_sk, uint64_t seed, uint64_t *ksk);
/* lwe_bootstrap_key_generation.rs:76- ; ggsw_encryption.rs:72-,300-334 ; layout [n][level 1..l][k+1][k+1][N] */
void orc_gen_bsk(const orc_params *p, const uint64_t *small_sk, const uint64_t *glwe_sk, uint64_t seed, uint64_t *bsk);
/* lwe_multi_bit_bootstrap_key_generation.rs:87-,401-427 ; layout [n/g][2^g][level][k+1][k+1][N] */
void orc_gen_multi_bit_bsk(const orc_params *p, const uint64_t *small_sk, const uint64_t *glwe_sk, uint64_t seed, uint64_t *bsk);
size_t orc_ksk_len(const orc_params *p);
size_t orc_bsk_len(const orc_params *p); /* classic or multi-bit depending on grouping_factor */

/* integer primitives -------------------------------------------------------------------------- */
uint64_t orc_closest_representable(uint64_t x, uint32_t base_log, uint32_t level);   /* decomposer.rs:98-118 */
uint32_t orc_closest_representable_u32(uint32_t x, uint32_t base_log, uint32_t level);
/* decomposer.rs:144-152 + iter.rs:37-50,120-127; digits[0] is level `level`, digits[level-1] is level 1 */
void orc_decompose(uint64_t x, uint32_t base_log, uint32_t level, int64_t *digits);
uint64_t orc_modulus_switch(uint64_t x, uint32_t log2_poly_size);                    /* fft_impl/common.rs:26-43 */
void orc_monomial_div(uint64_t *out, const uint64_t *in, size_t N, size_t degree);   /* polynomial_algorithms.rs:315-366 */
void orc_monomial_mul(uint64_t *out, const uint64_t *in, size_t N, size_t degree);   /* polynomial_algorithms.rs:219-270 */
void orc_monomial_mul_and_subtract(uint64_t *out, const uint64_t *in, size_t N, size_t degree); /* :425-497 */
void orc_sample_extract0(const orc_params *p, const uint64_t *glwe, uint64_t *lwe);  /* glwe_sample_extraction.rs:91-147 */
void orc_keyswitch(const orc_params *p, const uint64_t *ksk, const uint64_t *in, uint64_t *out); /* lwe_keyswitch.rs:96-170 */

/* shortint layer ------------------------------------------------------------------------------ */
/* engine/mod.rs:72-128; table[i] = f(i) for i < msg_mod*carry_mod; returns max f (the degree) */
uint64_t orc_fill_accumulator(const orc_params *p, const uint64_t *table, uint64_t *acc);
/* server_key/mod.rs:763-781 */
uint64_t orc_trivial_pbs(const orc_params *p, uint64_t body, const uint64_t *acc);
uint64_t orc_encode(const orc_params *p, uint64_t msg);                               /* client_side.rs:58-85 */
uint64_t orc_decode(const orc_params *p, uint64_t plaintext);                         /* client_key/mod.rs:281-302 */

/* f64 FFT (fft64/math/fft/mod.rs; concrete-fft restated as an unordered radix-2 DIF/DIT pair) --- */
void orc_fft_forward_integer(size_t N, const uint64_t *poly, double *re, double *im); /* mod.rs:220-239,496-515 */
void orc_fft_forward_torus(size_t N, const uint64_t *poly, double *re, double *im);   /* mod.rs:197-218 */
void orc_fft_add_backward_torus(size_t N, uint64_t *poly, double *re, double *im);    /* mod.rs:285-326,539-557 (in place on re/im) */

/* Fourier bootstrap key (bootstrap.rs:26-64, lwe_bootstrap_key_conversion.rs:99-) */
typedef struct orc_fourier_bsk orc_fourier_bsk;
orc_fourier_bsk *orc_fourier_bsk_new(const orc_params *p, const uint64_t *bsk_std);
void orc_fourier_bsk_free(orc_fourier_bsk *f);

/* external product, acc += ggsw (x) glwe (ggsw.rs:477-598). f64 flavour and exact-integer flavour. */
void orc_add_external_product_f64(const orc_params *p, const orc_fourier_bsk *f, size_t ggsw_index,
                                  uint64_t *out_glwe, const uint64_t *glwe);
void orc_add_external_product_exact(const orc_params *p, const uint64_t *ggsw_std,
                                    uint64_t *out_glwe, const uint64_t *glwe);

/* PBS (bootstrap.rs:242-364 classic; lwe_multi_bit_programmable_bootstrapping.rs deterministic order).
 * lwe_in: n+1 words under the small key; acc: (k+1)*N LUT; lwe_out: k*N+1 words. */
void orc_pbs_f64(const orc_params *p, const orc_fourier_bsk *f, const uint64_t *lwe_in, const uint64_t *acc, uint64_t *lwe_out);
/* test hook mirroring tfhe_b200_pbs_batch_partial: stop after n_steps mask elements (classic) / groups (multi-bit) */
void orc_pbs_f64_partial(const orc_params *p, const orc_fourier_bsk *f, const uint64_t *lwe_in, const uint64_t *acc, uint64_t *lwe_out,
                         size_t n_steps);
void orc_pbs_exact(const orc_params *p, const uint64_t *bsk_std, const uint64_t *lwe_in, const uint64_t *acc, uint64_t *lwe_out);
/* Exact PBS for classic AND multi-bit keys, stopped after max_steps like orc_pbs_f64_partial (SIZE_MAX = whole rotation).  The
 * polynomial products iterate over the key's nonzero coefficients, O(N * nnz) each: sparse test keys make whole batches affordable. */
void orc_pbs_exact_steps(const orc_params *p, const uint64_t *bsk_std, const uint64_t *lwe_in, const uint64_t *acc, uint64_t *lwe_out,
                         size_t max_steps);
/* batches of the above (no keyswitch), one ciphertext per OpenMP thread; luts: n_luts * (k+1)*N, lut_idx per ct or NULL (LUT 0).
 * orc_pbs_f64_batch is the same over a Fourier key.  Both return the threads used. */
int orc_pbs_exact_batch(const orc_params *p, const uint64_t *bsk_std, const uint64_t *luts, const uint32_t *lut_idx,
                        const uint64_t *in, uint64_t *out, size_t batch, size_t max_steps, int threads);
int orc_pbs_f64_batch(const orc_params *p, const orc_fourier_bsk *f, const uint64_t *luts, const uint32_t *lut_idx,
                      const uint64_t *in, uint64_t *out, size_t batch, size_t max_steps, int threads);

/* shortint/server_key/mod.rs:783-857: batched KS -> PBS, one independent ciphertext per OpenMP thread
 * (same structure as benches/core_crypto/pbs_bench.rs:512-536).  luts: n_luts * (k+1)*N, lut_idx per ct.
 * ks_out (optional, may be NULL): batch * (n+1) keyswitched ciphertexts.  Returns threads used. */
int orc_ks_pbs_batch(const orc_params *p, const uint64_t *ksk, const orc_fourier_bsk *f,
                     const uint64_t *luts, const uint32_t *lut_idx,
                     const uint64_t *in, uint64_t *out, uint64_t *ks_out, size_t batch, int threads);
int orc_max_threads(void);

/* ---- seeded keys (csprng_oracle.c): concrete-csprng's AES-128 CTR table + tfhe's seeded_*_decompression.rs ---- */
const uint8_t *orc_aes_sbox(void);
void orc_aes128_expand_key(const uint8_t key[16], uint8_t rk[176]);
void orc_aes128_encrypt_block(const uint8_t rk[176], const uint8_t in[16], uint8_t out[16]);
void orc_csprng_table_bytes(const uint8_t seed[16], uint64_t first, uint8_t *out, size_t n);   /* table byte 16*A + b */
void orc_csprng_generate_bytes(const uint8_t seed[16], uint64_t skip, uint8_t *out, size_t n); /* a fresh generator's output */
void orc_csprng_mask_words(const uint8_t seed[16], uint64_t first_word, uint64_t *out, size_t n);
size_t orc_seeded_bsk_len(const orc_params *p);   /* body polynomials only: rows * N */
size_t orc_seeded_ksk_len(const orc_params *p);   /* one body per (input key bit, level) */
void orc_decompress_seeded_bsk(const orc_params *p, const uint8_t seed[16], const uint64_t *bodies, uint64_t *bsk_std);
void orc_decompress_seeded_ksk(const orc_params *p, const uint8_t seed[16], const uint64_t *bodies, uint64_t *ksk);
/* test-side key generation: the seeded key a client would have produced (same plaintexts and noise, masks from the stream) */
void orc_compress_bsk(const orc_params *p, const uint64_t *glwe_sk, const uint8_t seed[16], const uint64_t *bsk_std, uint64_t *bodies);
void orc_compress_ksk(const orc_params *p, const uint64_t *small_sk, const uint8_t seed[16], const uint64_t *ksk, uint64_t *bodies);

#ifdef __cplusplus
}
#endif
#endif
