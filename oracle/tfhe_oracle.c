/*
 * oracle/tfhe_oracle.c -- CPU restatement of the tfhe-rs 0.5.0 KS-PBS path (see tfhe_oracle.h).
 * TEST INFRASTRUCTURE ONLY: never linked into or called from the product path.
 * All reference citations are relative to /root/reference/tfhe/src/.
 */
#include "tfhe_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

typedef unsigned __int128 u128;

/* hot loops get AVX-512 / AVX2 / baseline clones picked at load time (the .so travels to the GPU box) */
#define ORC_CLONES __attribute__((target_clones("arch=x86-64-v4", "arch=x86-64-v3", "default")))

/* ------------------------------------------------------------------------------------------- */
/* parameters                                                                                  */
/* ------------------------------------------------------------------------------------------- */

/* shortint/parameters/mod.rs:703-717 */
void orc_params_message_2_carry_2_ks_pbs(orc_params *p) {
    p->lwe_dim = 742; p->glwe_dim = 1; p->poly_size = 2048;
    p->pbs_base_log = 23; p->pbs_level = 1; p->ks_base_log = 3; p->ks_level = 5;
    p->grouping_factor = 0; p->msg_mod = 4; p->carry_mod = 4;
    p->lwe_std = 0.000007069849454709433; p->glwe_std = 0.00000000000000029403601535432533;
}

/* shortint/parameters/multi_bit.rs:173-190 */
void orc_params_multi_bit_message_2_carry_2_group_3_ks_pbs(orc_params *p) {
    p->lwe_dim = 888; p->glwe_dim = 1; p->poly_size = 2048;
    p->pbs_base_log = 21; p->pbs_level = 1; p->ks_base_log = 7; p->ks_level = 2;
    p->grouping_factor = 3; p->msg_mod = 4; p->carry_mod = 4;
    p->lwe_std = 0.0000006125031601933181; p->glwe_std = 0.0000000000000003152931493498455;
}

/* Not a reference set: a tiny, nearly noise-free set so exhaustive CPU tests finish in milliseconds. */
void orc_params_toy(orc_params *p) {
    p->lwe_dim = 24; p->glwe_dim = 1; p->poly_size = 256;
    p->pbs_base_log = 23; p->pbs_level = 1; p->ks_base_log = 3; p->ks_level = 5;
    p->grouping_factor = 0; p->msg_mod = 4; p->carry_mod = 4;
    p->lwe_std = 1e-9; p->glwe_std = 1e-16;
}

/* ------------------------------------------------------------------------------------------- */
/* PRNG                                                                                        */
/* ------------------------------------------------------------------------------------------- */

static uint64_t splitmix64(uint64_t *x) {
    uint64_t z = (*x += 0x9E3779B97F4A7C15ULL);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

void orc_rng_seed(orc_rng *r, uint64_t seed) {
    uint64_t x = seed;
    for (int i = 0; i < 4; i++) r->s[i] = splitmix64(&x);
    r->has_spare = 0; r->spare = 0.0;
}

static inline uint64_t rotl64(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }

uint64_t orc_rng_u64(orc_rng *r) {
    uint64_t *s = r->s;
    const uint64_t result = rotl64(s[1] * 5, 7) * 9;
    const uint64_t t = s[1] << 17;
    s[2] ^= s[0]; s[3] ^= s[1]; s[1] ^= s[2]; s[0] ^= s[3];
    s[2] ^= t; s[3] = rotl64(s[3], 45);
    return result;
}

/* standard normal by Box-Muller (commons/math/random/gaussian.rs:17-50 uses the same transform) */
double orc_rng_gauss(orc_rng *r) {
    if (r->has_spare) { r->has_spare = 0; return r->spare; }
    double u, v, s;
    do {
        u = (double)(orc_rng_u64(r) >> 11) * (1.0 / 9007199254740992.0) * 2.0 - 1.0;
        v = (double)(orc_rng_u64(r) >> 11) * (1.0 / 9007199254740992.0) * 2.0 - 1.0;
        s = u * u + v * v;
    } while (s >= 1.0 || s == 0.0);
    double m = sqrt(-2.0 * log(s) / s);
    r->spare = v * m; r->has_spare = 1;
    return u * m;
}

/* commons/math/torus/mod.rs:72-78 (scalar from_torus: f64::round = half away from zero) */
static inline uint64_t from_torus_scalar(double x) {
    double fract = x - round(x);
    fract *= 18446744073709551616.0;
    fract = round(fract);
    return (uint64_t)(int64_t)fract;
}

/* fft/x86.rs:823-875 + mm256_cvtpd_epi64: the AVX path rounds half-to-even (_MM_FROUND_NINT) */
static inline uint64_t from_torus_nint(double x) {
    double fract = x - nearbyint(x);
    fract = nearbyint(fract * 18446744073709551616.0);
    return (uint64_t)(int64_t)fract;
}

static inline uint64_t gaussian_torus(orc_rng *r, double std) {
    return from_torus_scalar(orc_rng_gauss(r) * std);
}

/* ------------------------------------------------------------------------------------------- */
/* sizes                                                                                       */
/* ------------------------------------------------------------------------------------------- */

size_t orc_ksk_len(const orc_params *p) {
    return (size_t)p->glwe_dim * p->poly_size * p->ks_level * (p->lwe_dim + 1);
}

static size_t ggsw_len(const orc_params *p) {
    size_t k1 = p->glwe_dim + 1;
    return (size_t)p->pbs_level * k1 * k1 * p->poly_size;
}

size_t orc_bsk_len(const orc_params *p) {
    if (p->grouping_factor == 0) return (size_t)p->lwe_dim * ggsw_len(p);
    size_t groups = p->lwe_dim / p->grouping_factor;
    return groups * ((size_t)1 << p->grouping_factor) * ggsw_len(p);
}

/* ------------------------------------------------------------------------------------------- */
/* keys, LWE / GLWE encryption                                                                 */
/* ------------------------------------------------------------------------------------------- */

void orc_gen_binary_key(orc_rng *r, uint64_t *sk, size_t len) {
    for (size_t i = 0; i < len; i++) sk[i] = orc_rng_u64(r) >> 63;
}

void orc_lwe_encrypt(const uint64_t *sk, size_t dim, uint64_t plaintext, double std, orc_rng *r, uint64_t *ct) {
    uint64_t body = plaintext + gaussian_torus(r, std);
    for (size_t i = 0; i < dim; i++) {
        ct[i] = orc_rng_u64(r);
        body += ct[i] * sk[i];
    }
    ct[dim] = body;
}

uint64_t orc_lwe_decrypt(const uint64_t *sk, size_t dim, const uint64_t *ct) {
    uint64_t acc = ct[dim];
    for (size_t i = 0; i < dim; i++) acc -= ct[i] * sk[i];
    return acc;
}

/* lwe_keyswitch_key_generation.rs:107-129: for input key bit s_i, levels stored l..1, plaintext of
 * level j = s_i << (64 - base_log*j) (term.rs:50-53), encrypted under the OUTPUT (small) key. */
void orc_gen_ksk(const orc_params *p, const uint64_t *big_sk, const uint64_t *small_sk, uint64_t seed, uint64_t *ksk) {
    size_t in_dim = (size_t)p->glwe_dim * p->poly_size, n = p->lwe_dim, L = p->ks_level;
    #pragma omp parallel for schedule(static)
    for (long i = 0; i < (long)in_dim; i++) {
        orc_rng r; orc_rng_seed(&r, seed ^ (0x4B534B00ULL + (uint64_t)i * 0x100000001B3ULL));
        for (size_t idx = 0; idx < L; idx++) {
            uint32_t level = (uint32_t)(L - idx); /* stored level L first */
            uint64_t pt = big_sk[i] << (64 - p->ks_base_log * level);
            orc_lwe_encrypt(small_sk, n, pt, p->lwe_std, &r, ksk + ((size_t)i * L + idx) * (n + 1));
        }
    }
}

/* body += mask_poly * key_poly in Z_2^64[X]/(X^N+1) for a BINARY key polynomial */
static void negacyclic_mul_binary_add(uint64_t *body, const uint64_t *mask, const uint64_t *key, size_t N) {
    for (size_t t = 0; t < N; t++) {
        if (!key[t]) continue;
        for (size_t j = 0; j < N - t; j++) body[j + t] += mask[j];
        for (size_t j = N - t; j < N; j++) body[j + t - N] -= mask[j];
    }
}

/* glwe_encryption.rs:136-171: body = sum_i mask_i * S_i + plaintext(already in body) + e */
static void glwe_encrypt_assign(const orc_params *p, const uint64_t *glwe_sk, uint64_t *glwe, orc_rng *r) {
    size_t N = p->poly_size, k = p->glwe_dim;
    uint64_t *body = glwe + k * N;
    for (size_t i = 0; i < k; i++) {
        uint64_t *mask = glwe + i * N;
        for (size_t j = 0; j < N; j++) mask[j] = orc_rng_u64(r);
        negacyclic_mul_binary_add(body, mask, glwe_sk + i * N, N);
    }
    for (size_t j = 0; j < N; j++) body[j] += gaussian_torus(r, p->glwe_std);
}

/* ggsw_encryption.rs:117-126 (factor = -m * 2^(64 - base_log*level), levels stored 1..l) and
 * :300-334 (row r<k: body = factor * S_r(X); last row: body[0] = -factor). */
static void ggsw_encrypt_constant(const orc_params *p, const uint64_t *glwe_sk, uint64_t m, uint64_t *ggsw, orc_rng *r) {
    size_t N = p->poly_size, k = p->glwe_dim, k1 = k + 1;
    for (uint32_t level = 1; level <= p->pbs_level; level++) {
        uint64_t factor = (uint64_t)0 - (m << (64 - p->pbs_base_log * level));
        for (size_t row = 0; row < k1; row++) {
            uint64_t *glwe = ggsw + (((size_t)(level - 1) * k1 + row) * k1) * N;
            uint64_t *body = glwe + k * N;
            if (row < k) {
                for (size_t j = 0; j < N; j++) body[j] = glwe_sk[row * N + j] * factor;
            } else {
                memset(body, 0, N * sizeof(uint64_t));
                body[0] = (uint64_t)0 - factor;
            }
            glwe_encrypt_assign(p, glwe_sk, glwe, r);
        }
    }
}

void orc_gen_bsk(const orc_params *p, const uint64_t *small_sk, const uint64_t *glwe_sk, uint64_t seed, uint64_t *bsk) {
    size_t gl = ggsw_len(p);
    #pragma omp parallel for schedule(dynamic, 4)
    for (long i = 0; i < (long)p->lwe_dim; i++) {
        orc_rng r; orc_rng_seed(&r, seed ^ (0x42534B00ULL + (uint64_t)i * 0x100000001B3ULL));
        ggsw_encrypt_constant(p, glwe_sk, small_sk[i], bsk + (size_t)i * gl, &r);
    }
}

/* lwe_multi_bit_bootstrap_key_generation.rs:401-427 combine_key_bits */
static uint64_t combine_key_bits(size_t bit_selector, const uint64_t *key_elems, size_t g) {
    uint64_t prod = 1;
    for (size_t bit_idx = 0; bit_idx < g; bit_idx++) {
        size_t bit_position = g - (bit_idx + 1);
        uint64_t inversion_bit = ((bit_selector >> bit_position) & 1) ^ 1;
        prod *= key_elems[bit_idx] ^ inversion_bit;
    }
    return prod;
}

void orc_gen_multi_bit_bsk(const orc_params *p, const uint64_t *small_sk, const uint64_t *glwe_sk, uint64_t seed, uint64_t *bsk) {
    size_t gl = ggsw_len(p), g = p->grouping_factor, per = (size_t)1 << g, groups = p->lwe_dim / g;
    #pragma omp parallel for schedule(dynamic, 2)
    for (long t = 0; t < (long)(groups * per); t++) {
        size_t grp = (size_t)t / per, sel = (size_t)t % per;
        orc_rng r; orc_rng_seed(&r, seed ^ (0x4D42534BULL + (uint64_t)t * 0x100000001B3ULL));
        uint64_t m = combine_key_bits(sel, small_sk + grp * g, g);
        ggsw_encrypt_constant(p, glwe_sk, m, bsk + (size_t)t * gl, &r);
    }
}

/* ------------------------------------------------------------------------------------------- */
/* integer primitives                                                                          */
/* ------------------------------------------------------------------------------------------- */

/* commons/math/decomposition/decomposer.rs:98-118 */
uint64_t orc_closest_representable(uint64_t x, uint32_t base_log, uint32_t level) {
    uint32_t non_rep = 64 - base_log * level;
    uint32_t shift = non_rep - 1;
    uint64_t res = x >> shift;
    res += 1;
    res &= ~(uint64_t)1;
    return res << shift;
}

uint32_t orc_closest_representable_u32(uint32_t x, uint32_t base_log, uint32_t level) {
    uint32_t non_rep = 32 - base_log * level;
    uint32_t shift = non_rep - 1;
    uint32_t res = x >> shift;
    res += 1;
    res &= ~(uint32_t)1;
    return res << shift;
}

/* commons/math/decomposition/iter.rs:120-127 */
static inline __attribute__((always_inline)) uint64_t decompose_one_level(uint32_t base_log, uint64_t *state, uint64_t mod_b_mask) {
    uint64_t res = *state & mod_b_mask;
    *state >>= base_log;
    uint64_t carry = ((res - 1) | *state) & res;
    carry >>= base_log - 1;
    *state += carry;
    return res - (carry << base_log);
}

/* decomposer.rs:144-152 + iter.rs:37-50: yields level `level` first, level 1 last */
void orc_decompose(uint64_t x, uint32_t base_log, uint32_t level, int64_t *digits) {
    uint64_t state = orc_closest_representable(x, base_log, level) >> (64 - base_log * level);
    uint64_t mask = ((uint64_t)1 << base_log) - 1;
    for (uint32_t i = 0; i < level; i++) digits[i] = (int64_t)decompose_one_level(base_log, &state, mask);
}

/* fft_impl/common.rs:26-43 with offset 0, lut_count_log 0 */
uint64_t orc_modulus_switch(uint64_t x, uint32_t log2_poly_size) {
    uint64_t out = x >> (64 - log2_poly_size - 2);
    out += 1;
    out >>= 1;
    return out;
}

/* polynomial_algorithms.rs:315-366 */
ORC_CLONES
void orc_monomial_div(uint64_t *out, const uint64_t *in, size_t N, size_t degree) {
    size_t rem = degree % N, cycles = degree / N;
    if (cycles % 2 == 0) {
        for (size_t j = 0; j < N - rem; j++) out[j] = in[j + rem];
        for (size_t j = 0; j < rem; j++) out[N - rem + j] = (uint64_t)0 - in[j];
    } else {
        for (size_t j = 0; j < N - rem; j++) out[j] = (uint64_t)0 - in[j + rem];
        for (size_t j = 0; j < rem; j++) out[N - rem + j] = in[j];
    }
}

/* polynomial_algorithms.rs:219-270 */
void orc_monomial_mul(uint64_t *out, const uint64_t *in, size_t N, size_t degree) {
    size_t rem = degree % N, cycles = degree / N;
    if (cycles % 2 == 0) {
        for (size_t j = 0; j < rem; j++) out[j] = (uint64_t)0 - in[N - rem + j];
        for (size_t j = rem; j < N; j++) out[j] = in[j - rem];
    } else {
        for (size_t j = 0; j < rem; j++) out[j] = in[N - rem + j];
        for (size_t j = rem; j < N; j++) out[j] = (uint64_t)0 - in[j - rem];
    }
}

/* polynomial_algorithms.rs:425-497: out = in * X^degree - in */
ORC_CLONES
void orc_monomial_mul_and_subtract(uint64_t *out, const uint64_t *in, size_t N, size_t degree) {
    size_t rem = degree % N, cycles = degree / N;
    if (cycles % 2 == 0) {
        for (size_t j = 0; j < rem; j++) out[j] = ((uint64_t)0 - in[N - rem + j]) - in[j];
        for (size_t j = rem; j < N; j++) out[j] = in[j - rem] - in[j];
    } else {
        for (size_t j = 0; j < rem; j++) out[j] = in[N - rem + j] - in[j];
        for (size_t j = rem; j < N; j++) out[j] = ((uint64_t)0 - in[j - rem]) - in[j];
    }
}

/* glwe_sample_extraction.rs:125-146 with nth = 0: body = B[0]; per mask poly: reverse, negate the
 * first N-1 (after reversal: all but the one that came from A[0]), rotate so A[0] is first. */
void orc_sample_extract0(const orc_params *p, const uint64_t *glwe, uint64_t *lwe) {
    size_t N = p->poly_size, k = p->glwe_dim;
    for (size_t i = 0; i < k; i++) {
        const uint64_t *A = glwe + i * N;
        uint64_t *o = lwe + i * N;
        o[0] = A[0];
        for (size_t j = 1; j < N; j++) o[j] = (uint64_t)0 - A[N - j];
    }
    lwe[k * N] = glwe[k * N];
}

/* lwe_keyswitch.rs:144-169 + slice_algorithms.rs:363-461 (lhs[j] -= rhs[j] * digit, wrapping) */
ORC_CLONES
void orc_keyswitch(const orc_params *p, const uint64_t *ksk, const uint64_t *in, uint64_t *out) {
    size_t in_dim = (size_t)p->glwe_dim * p->poly_size, n = p->lwe_dim, L = p->ks_level;
    int64_t digits[64];
    memset(out, 0, (n + 1) * sizeof(uint64_t));
    out[n] = in[in_dim];
    for (size_t i = 0; i < in_dim; i++) {
        orc_decompose(in[i], p->ks_base_log, p->ks_level, digits);
        for (size_t idx = 0; idx < L; idx++) {
            uint64_t d = (uint64_t)digits[idx];
            if (d == 0) continue;
            const uint64_t *row = ksk + (i * L + idx) * (n + 1);
            for (size_t j = 0; j <= n; j++) out[j] -= row[j] * d;
        }
    }
}

/* ------------------------------------------------------------------------------------------- */
/* shortint layer                                                                              */
/* ------------------------------------------------------------------------------------------- */

uint64_t orc_encode(const orc_params *p, uint64_t msg) {
    uint64_t delta = ((uint64_t)1 << 63) / (p->msg_mod * p->carry_mod);
    return msg * delta;
}

uint64_t orc_decode(const orc_params *p, uint64_t plaintext) {
    uint64_t delta = ((uint64_t)1 << 63) / (p->msg_mod * p->carry_mod);
    uint64_t rounding_bit = delta >> 1;
    uint64_t rounding = (plaintext & rounding_bit) << 1;
    return (plaintext + rounding) / delta;
}

uint64_t orc_fill_accumulator(const orc_params *p, const uint64_t *table, uint64_t *acc) {
    size_t N = p->poly_size, k = p->glwe_dim;
    size_t modulus_sup = (size_t)p->msg_mod * p->carry_mod;
    size_t box = N / modulus_sup, half = box / 2;
    uint64_t delta = ((uint64_t)1 << 63) / modulus_sup;
    uint64_t max_value = 0;
    memset(acc, 0, k * N * sizeof(uint64_t));
    uint64_t *body = acc + k * N;
    uint64_t *tmp = (uint64_t *)malloc(N * sizeof(uint64_t));
    for (size_t i = 0; i < modulus_sup; i++) {
        uint64_t f = table[i];
        if (f > max_value) max_value = f;
        for (size_t j = 0; j < box; j++) tmp[i * box + j] = f * delta;
    }
    for (size_t j = 0; j < half; j++) tmp[j] = (uint64_t)0 - tmp[j];
    for (size_t j = 0; j < N; j++) body[j] = tmp[(j + half) % N]; /* rotate_left(half) */
    free(tmp);
    return max_value;
}

uint64_t orc_trivial_pbs(const orc_params *p, uint64_t body_in, const uint64_t *acc) {
    size_t N = p->poly_size, k = p->glwe_dim;
    uint64_t modulus_sup = (uint64_t)p->msg_mod * p->carry_mod;
    uint64_t delta = ((uint64_t)1 << 63) / modulus_sup;
    uint64_t ct_value = body_in / delta;
    size_t box = N / modulus_sup;
    const uint64_t *body = acc + k * N;
    if (ct_value >= modulus_sup) {
        ct_value %= modulus_sup;
        return (uint64_t)0 - body[ct_value * box];
    }
    return body[ct_value * box];
}

/* ------------------------------------------------------------------------------------------- */
/* f64 negacyclic FFT: fold + twist + size-N/2 complex FFT (fft64/math/fft/mod.rs; eprint 2021/480) */
/* concrete-fft's unordered plan is restated as a radix-2 DIF forward (natural in, bit-reversed */
/* out) and radix-2 DIT inverse (bit-reversed in, natural out); only pointwise products happen  */
/* in between, so any self-consistent ordering gives the same polynomial product.                */
/* ------------------------------------------------------------------------------------------- */

#define ORC_MAX_LOG_N 15
/* Four-step layout: M = N/2 = R*C, index j = r*C + c.  Forward: radix-2 DIF down the R rows (every
 * butterfly is a vector operation over the C contiguous columns), twiddle by W_M^(c*q), transpose,
 * radix-2 DIF down the C rows.  Output order is a fixed permutation (bit-reversed digits), which is
 * all the external product needs.  The inverse undoes each step with conjugate twiddles. */
typedef struct {
    size_t N, R, C;
    double *tw_re, *tw_im;   /* Twisties (mod.rs:58-69): w_j = exp(i*pi*j/N), j < N/2 */
    double *sr_re, *sr_im;   /* stage twiddles for length-R DIF: at offset h, exp(-2*pi*i*j/(2h)), j<h */
    double *sc_re, *sc_im;   /* same for length C */
    double *x_re, *x_im;     /* inter-pass twiddles [rho][c] = W_M^(c * brev_R(rho)) */
} fft_plan;

static fft_plan g_plans[ORC_MAX_LOG_N + 1];

static size_t brev(size_t x, int bits) {
    size_t r = 0;
    for (int i = 0; i < bits; i++) r |= ((x >> i) & 1) << (bits - 1 - i);
    return r;
}

static void make_stage_tw(size_t len, double **re, double **im) {
    double *a = (double *)malloc(len * sizeof(double)), *b = (double *)malloc(len * sizeof(double));
    a[0] = 1.0; b[0] = 0.0;
    for (size_t h = 1; h < len; h <<= 1)
        for (size_t j = 0; j < h; j++) {
            long double ang = -3.14159265358979323846264338327950288L * (long double)j / (long double)h;
            a[h + j] = (double)cosl(ang); b[h + j] = (double)sinl(ang);
        }
    *re = a; *im = b;
}

static const fft_plan *get_plan(size_t N) {
    int lg = 0;
    while (((size_t)1 << lg) < N) lg++;
    fft_plan *pl = &g_plans[lg];
    if (pl->N == N) return pl;
    #pragma omp critical(orc_plan)
    {
        if (pl->N != N) {
            size_t M = N / 2;
            int lgM = lg - 1, lgR = lgM / 2, lgC = lgM - lgR;
            size_t R = (size_t)1 << lgR, C = (size_t)1 << lgC;
            double *tw_re = (double *)malloc(M * sizeof(double)), *tw_im = (double *)malloc(M * sizeof(double));
            for (size_t j = 0; j < M; j++) {
                long double a = 3.14159265358979323846264338327950288L * (long double)j / (long double)N;
                tw_re[j] = (double)cosl(a); tw_im[j] = (double)sinl(a);
            }
            make_stage_tw(R, &pl->sr_re, &pl->sr_im);
            make_stage_tw(C, &pl->sc_re, &pl->sc_im);
            pl->x_re = (double *)malloc(M * sizeof(double)); pl->x_im = (double *)malloc(M * sizeof(double));
            for (size_t rho = 0; rho < R; rho++)
                for (size_t c = 0; c < C; c++) {
                    size_t e = (c * brev(rho, lgR)) % M;
                    long double a = -2.0L * 3.14159265358979323846264338327950288L * (long double)e / (long double)M;
                    pl->x_re[rho * C + c] = (double)cosl(a); pl->x_im[rho * C + c] = (double)sinl(a);
                }
            pl->tw_re = tw_re; pl->tw_im = tw_im; pl->R = R; pl->C = C;
            #pragma omp flush
            pl->N = N;
        }
    }
    return pl;
}


/* radix-2 DIF over `rows` rows of `cols` contiguous elements */
ORC_CLONES
static void dif_rows(double *restrict re, double *restrict im, size_t rows, size_t cols,
                     const double *restrict sw_re, const double *restrict sw_im) {
    for (size_t h = rows / 2; h >= 1; h >>= 1)
        for (size_t b = 0; b < rows; b += 2 * h)
            for (size_t j = 0; j < h; j++) {
                double wr = sw_re[h + j], wi = sw_im[h + j];
                double *restrict ar = re + (b + j) * cols, *restrict ai = im + (b + j) * cols;
                double *restrict cr = re + (b + j + h) * cols, *restrict ci = im + (b + j + h) * cols;
                for (size_t c = 0; c < cols; c++) {
                    double xr = ar[c], xi = ai[c], yr = cr[c], yi = ci[c];
                    double dr = xr - yr, di = xi - yi;
                    ar[c] = xr + yr; ai[c] = xi + yi;
                    cr[c] = dr * wr - di * wi;
                    ci[c] = dr * wi + di * wr;
                }
            }
}

/* exact inverse of dif_rows up to a factor `rows` (radix-2 DIT, conjugate twiddles) */
ORC_CLONES
static void dit_rows_inv(double *restrict re, double *restrict im, size_t rows, size_t cols,
                         const double *restrict sw_re, const double *restrict sw_im) {
    for (size_t h = 1; h < rows; h <<= 1)
        for (size_t b = 0; b < rows; b += 2 * h)
            for (size_t j = 0; j < h; j++) {
                double wr = sw_re[h + j], wi = sw_im[h + j];
                double *restrict ar = re + (b + j) * cols, *restrict ai = im + (b + j) * cols;
                double *restrict cr = re + (b + j + h) * cols, *restrict ci = im + (b + j + h) * cols;
                for (size_t c = 0; c < cols; c++) {
                    double yr = cr[c] * wr + ci[c] * wi;
                    double yi = ci[c] * wr - cr[c] * wi;
                    double xr = ar[c], xi = ai[c];
                    ar[c] = xr + yr; ai[c] = xi + yi;
                    cr[c] = xr - yr; ci[c] = xi - yi;
                }
            }
}

ORC_CLONES
static void twiddle_transpose(const fft_plan *pl, double *restrict re, double *restrict im, int inverse) {
    size_t R = pl->R, C = pl->C, M = R * C;
    double tr[M], ti[M];
    if (!inverse) { /* [rho][c] * x -> [c][rho] */
        for (size_t rho = 0; rho < R; rho++)
            for (size_t c = 0; c < C; c++) {
                double a = re[rho * C + c], b = im[rho * C + c], wr = pl->x_re[rho * C + c], wi = pl->x_im[rho * C + c];
                tr[c * R + rho] = a * wr - b * wi;
                ti[c * R + rho] = a * wi + b * wr;
            }
    } else {        /* [c][rho] -> [rho][c] * conj(x) */
        for (size_t c = 0; c < C; c++)
            for (size_t rho = 0; rho < R; rho++) {
                double a = re[c * R + rho], b = im[c * R + rho], wr = pl->x_re[rho * C + c], wi = pl->x_im[rho * C + c];
                tr[rho * C + c] = a * wr + b * wi;
                ti[rho * C + c] = b * wr - a * wi;
            }
    }
    memcpy(re, tr, M * sizeof(double)); memcpy(im, ti, M * sizeof(double));
}

static void fft_dif(const fft_plan *pl, double *re, double *im) {
    dif_rows(re, im, pl->R, pl->C, pl->sr_re, pl->sr_im);
    twiddle_transpose(pl, re, im, 0);
    dif_rows(re, im, pl->C, pl->R, pl->sc_re, pl->sc_im);
}

static void fft_dit_inv(const fft_plan *pl, double *re, double *im) {
    dit_rows_inv(re, im, pl->C, pl->R, pl->sc_re, pl->sc_im);
    twiddle_transpose(pl, re, im, 1);
    dit_rows_inv(re, im, pl->R, pl->C, pl->sr_re, pl->sr_im);
}

/* mod.rs:220-239 convert_forward_integer_scalar (input as SIGNED i64 -> f64), then plan.fwd (:513) */
ORC_CLONES
void orc_fft_forward_integer(size_t N, const uint64_t *poly, double *re, double *im) {
    const fft_plan *pl = get_plan(N);
    size_t M = N / 2;
    for (size_t j = 0; j < M; j++) {
        double a = (double)(int64_t)poly[j], b = (double)(int64_t)poly[j + M];
        re[j] = a * pl->tw_re[j] - b * pl->tw_im[j];
        im[j] = a * pl->tw_im[j] + b * pl->tw_re[j];
    }
    fft_dif(pl, re, im);
}

/* mod.rs:197-218 convert_forward_torus (signed * 2^-64) */
ORC_CLONES
void orc_fft_forward_torus(size_t N, const uint64_t *poly, double *re, double *im) {
    const fft_plan *pl = get_plan(N);
    size_t M = N / 2;
    const double norm = 5.421010862427522e-20; /* 2^-64 */
    for (size_t j = 0; j < M; j++) {
        double a = (double)(int64_t)poly[j] * norm, b = (double)(int64_t)poly[j + M] * norm;
        re[j] = a * pl->tw_re[j] - b * pl->tw_im[j];
        im[j] = a * pl->tw_im[j] + b * pl->tw_re[j];
    }
    fft_dif(pl, re, im);
}

/* mod.rs:539-557 plan.inv then :285-326 convert_add_backward_torus: multiply by conj(w_j)/(N/2),
 * from_torus, wrapping add.  Rounding follows the x86 path the reference actually runs (half-to-even). */
ORC_CLONES
void orc_fft_add_backward_torus(size_t N, uint64_t *poly, double *re, double *im) {
    const fft_plan *pl = get_plan(N);
    size_t M = N / 2;
    fft_dit_inv(pl, re, im);
    double norm = 1.0 / (double)M;
    for (size_t j = 0; j < M; j++) {
        double wr = pl->tw_re[j] * norm, wi = pl->tw_im[j] * norm;
        double tr = re[j] * wr + im[j] * wi;
        double ti = im[j] * wr - re[j] * wi;
        poly[j] += from_torus_nint(tr);
        poly[j + M] += from_torus_nint(ti);
    }
}

/* ------------------------------------------------------------------------------------------- */
/* Fourier BSK                                                                                  */
/* ------------------------------------------------------------------------------------------- */

struct orc_fourier_bsk {
    orc_params p;
    size_t n_ggsw;     /* n (classic) or (n/g)*2^g (multi-bit) */
    size_t ggsw_polys; /* level*(k+1)*(k+1) */
    double *re, *im;   /* [n_ggsw][level 1..l][row][col][N/2] */
};

orc_fourier_bsk *orc_fourier_bsk_new(const orc_params *p, const uint64_t *bsk_std) {
    orc_fourier_bsk *f = (orc_fourier_bsk *)calloc(1, sizeof(*f));
    size_t N = p->poly_size, M = N / 2, k1 = p->glwe_dim + 1;
    f->p = *p;
    f->ggsw_polys = (size_t)p->pbs_level * k1 * k1;
    f->n_ggsw = orc_bsk_len(p) / (f->ggsw_polys * N);
    size_t total = f->n_ggsw * f->ggsw_polys;
    f->re = (double *)aligned_alloc(64, total * M * sizeof(double));
    f->im = (double *)aligned_alloc(64, total * M * sizeof(double));
    (void)get_plan(N);
    #pragma omp parallel for schedule(static)
    for (long t = 0; t < (long)total; t++)
        orc_fft_forward_torus(N, bsk_std + (size_t)t * N, f->re + (size_t)t * M, f->im + (size_t)t * M);
    return f;
}

void orc_fourier_bsk_free(orc_fourier_bsk *f) {
    if (!f) return;
    free(f->re); free(f->im); free(f);
}

/* ------------------------------------------------------------------------------------------- */
/* external product                                                                             */
/* ------------------------------------------------------------------------------------------- */

/* scratch for one PBS */
typedef struct {
    size_t N, k1, L;
    uint64_t *states;          /* k1*N decomposition states */
    uint64_t *digits;          /* k1*N current-level digits */
    double *f_re, *f_im;       /* N/2 */
    double *o_re, *o_im;       /* k1 * N/2 */
    double *g_re, *g_im;       /* combined multi-bit ggsw: L*k1*k1*N/2 */
    double *m_re, *m_im;       /* monomial spectrum N/2 */
    uint64_t *ct0, *ct1, *mono;
} pbs_scratch;

static void scratch_init(pbs_scratch *s, const orc_params *p) {
    size_t N = p->poly_size, M = N / 2, k1 = p->glwe_dim + 1, L = p->pbs_level;
    s->N = N; s->k1 = k1; s->L = L;
    s->states = (uint64_t *)malloc(k1 * N * 8); s->digits = (uint64_t *)malloc(k1 * N * 8);
    s->f_re = (double *)aligned_alloc(64, M * 8); s->f_im = (double *)aligned_alloc(64, M * 8);
    s->o_re = (double *)aligned_alloc(64, k1 * M * 8); s->o_im = (double *)aligned_alloc(64, k1 * M * 8);
    s->g_re = (double *)aligned_alloc(64, L * k1 * k1 * M * 8); s->g_im = (double *)aligned_alloc(64, L * k1 * k1 * M * 8);
    s->m_re = (double *)aligned_alloc(64, M * 8); s->m_im = (double *)aligned_alloc(64, M * 8);
    s->ct0 = (uint64_t *)malloc(k1 * N * 8); s->ct1 = (uint64_t *)malloc(k1 * N * 8);
    s->mono = (uint64_t *)malloc(N * 8);
}

static void scratch_free(pbs_scratch *s) {
    free(s->states); free(s->digits); free(s->f_re); free(s->f_im); free(s->o_re); free(s->o_im);
    free(s->g_re); free(s->g_im); free(s->m_re); free(s->m_im); free(s->ct0); free(s->ct1); free(s->mono);
}

ORC_CLONES
static void cmul_acc(double *restrict or_, double *restrict oi, const double *restrict gr, const double *restrict gi,
                     const double *restrict fr, const double *restrict fi, size_t M, int init) {
    if (init) for (size_t j = 0; j < M; j++) { or_[j] = gr[j] * fr[j] - gi[j] * fi[j]; oi[j] = gr[j] * fi[j] + gi[j] * fr[j]; }
    else for (size_t j = 0; j < M; j++) { or_[j] += gr[j] * fr[j] - gi[j] * fi[j]; oi[j] += gr[j] * fi[j] + gi[j] * fr[j]; }
}

/* ggsw.rs:477-598 with the Fourier GGSW given as SoA planes [level 1..l][row][col][N/2] */
ORC_CLONES
static void add_external_product_f64_planes(const orc_params *p, const double *g_re, const double *g_im,
                                            uint64_t *out, const uint64_t *glwe, pbs_scratch *s) {
    size_t N = p->poly_size, M = N / 2, k1 = p->glwe_dim + 1, L = p->pbs_level;
    uint32_t bl = p->pbs_base_log;
    uint64_t mask = ((uint64_t)1 << bl) - 1;
    /* math/decomposition.rs:25-44: states = closest_representable(x) >> (64 - bl*L) */
    for (size_t j = 0; j < k1 * N; j++)
        s->states[j] = orc_closest_representable(glwe[j], bl, p->pbs_level) >> (64 - bl * L);
    int init = 1;
    for (size_t lv = L; lv >= 1; lv--) { /* ggsw.into_levels().rev(): level L first (:524) */
        for (size_t j = 0; j < k1 * N; j++) s->digits[j] = decompose_one_level(bl, &s->states[j], mask);
        for (size_t row = 0; row < k1; row++) {
            orc_fft_forward_integer(N, s->digits + row * N, s->f_re, s->f_im);
            for (size_t col = 0; col < k1; col++) {
                size_t off = (((lv - 1) * k1 + row) * k1 + col) * M;
                cmul_acc(s->o_re + col * M, s->o_im + col * M, g_re + off, g_im + off, s->f_re, s->f_im, M, init);
            }
            init = 0;
        }
    }
    for (size_t col = 0; col < k1; col++)
        orc_fft_add_backward_torus(N, out + col * N, s->o_re + col * M, s->o_im + col * M);
}

void orc_add_external_product_f64(const orc_params *p, const orc_fourier_bsk *f, size_t ggsw_index,
                                  uint64_t *out_glwe, const uint64_t *glwe) {
    pbs_scratch s; scratch_init(&s, p);
    size_t M = p->poly_size / 2;
    size_t off = ggsw_index * f->ggsw_polys * M;
    add_external_product_f64_planes(p, f->re + off, f->im + off, out_glwe, glwe, &s);
    scratch_free(&s);
}

/* Exact flavour: the same decomposition, but the polynomial products are exact negacyclic
 * convolutions in Z_2^64 (the torus) -- independent of any FFT. */
void orc_add_external_product_exact(const orc_params *p, const uint64_t *ggsw_std, uint64_t *out, const uint64_t *glwe) {
    size_t N = p->poly_size, k1 = p->glwe_dim + 1, L = p->pbs_level;
    uint32_t bl = p->pbs_base_log;
    uint64_t mask = ((uint64_t)1 << bl) - 1;
    uint64_t *states = (uint64_t *)malloc(k1 * N * 8);
    uint64_t *digits = (uint64_t *)malloc(N * 8);
    for (size_t j = 0; j < k1 * N; j++)
        states[j] = orc_closest_representable(glwe[j], bl, p->pbs_level) >> (64 - bl * L);
    for (size_t lv = L; lv >= 1; lv--) {
        for (size_t row = 0; row < k1; row++) {
            for (size_t j = 0; j < N; j++) digits[j] = decompose_one_level(bl, &states[row * N + j], mask);
            for (size_t col = 0; col < k1; col++) {
                const uint64_t *g = ggsw_std + ((((lv - 1) * k1 + row) * k1) + col) * N;
                uint64_t *o = out + col * N;
                for (size_t a = 0; a < N; a++) {
                    uint64_t d = digits[a];
                    if (!d) continue;
                    for (size_t b = 0; b < N - a; b++) o[a + b] += d * g[b];
                    for (size_t b = N - a; b < N; b++) o[a + b - N] -= d * g[b];
                }
            }
        }
    }
    free(states); free(digits);
}

/* ------------------------------------------------------------------------------------------- */
/* PBS                                                                                          */
/* ------------------------------------------------------------------------------------------- */

static uint32_t ilog2(size_t x) { uint32_t l = 0; while (((size_t)1 << l) < x) l++; return l; }

/* multi-bit: lwe_multi_bit_programmable_bootstrapping.rs:18-84 prepare_multi_bit_ggsw_mem_optimized */
static void prepare_multi_bit_ggsw(const orc_params *p, const orc_fourier_bsk *f, size_t group,
                                   const uint64_t *mask_elems, pbs_scratch *s) {
    size_t N = p->poly_size, M = N / 2, g = p->grouping_factor, per = (size_t)1 << g;
    size_t plane = f->ggsw_polys * M;
    const double *base_re = f->re + group * per * plane, *base_im = f->im + group * per * plane;
    memcpy(s->g_re, base_re, plane * 8); memcpy(s->g_im, base_im, plane * 8);
    uint32_t lgN = ilog2(N);
    for (size_t idx = 1; idx < per; idx++) {
        uint64_t deg = 0;
        for (size_t mi = 0; mi < g; mi++) {
            size_t pos = g - (mi + 1);
            deg += (uint64_t)((idx >> pos) & 1) * mask_elems[mi];
        }
        size_t sw = (size_t)orc_modulus_switch(deg, lgN);
        /* monomial spectrum (fft/mod.rs:408-445): transform of X^sw in Z[X]/(X^N+1) */
        memset(s->mono, 0, N * 8);
        size_t d = sw % N;
        s->mono[d] = ((sw / N) % 2 == 1) ? (uint64_t)0 - 1 : 1;
        orc_fft_forward_integer(N, s->mono, s->m_re, s->m_im);
        const double *gr = base_re + idx * plane, *gi = base_im + idx * plane;
        for (size_t q = 0; q < f->ggsw_polys; q++)
            cmul_acc(s->g_re + q * M, s->g_im + q * M, gr + q * M, gi + q * M, s->m_re, s->m_im, M, 0);
    }
}

/* max_steps bounds the number of mask elements (classic) / groups (multi-bit) that are processed: the test hook behind
 * orc_pbs_f64_partial, mirroring tfhe_b200_pbs_batch_partial; SIZE_MAX = the whole blind rotation */
static void blind_rotate_f64_steps(const orc_params *p, const orc_fourier_bsk *f, const uint64_t *lwe_in,
                                   pbs_scratch *s, size_t max_steps) {
    size_t N = p->poly_size, M = N / 2, k1 = p->glwe_dim + 1, n = p->lwe_dim;
    uint32_t lgN = ilog2(N);
    size_t plane = f->ggsw_polys * M;
    /* bootstrap.rs:254-271: acc <- acc * X^{-b_hat}; ct0 holds a copy of the LUT on entry */
    size_t b_hat = (size_t)orc_modulus_switch(lwe_in[n], lgN);
    for (size_t q = 0; q < k1; q++) orc_monomial_div(s->ct1 + q * N, s->ct0 + q * N, N, b_hat);
    memcpy(s->ct0, s->ct1, k1 * N * 8);
    if (p->grouping_factor == 0) {
        for (size_t i = 0; i < n && i < max_steps; i++) { /* bootstrap.rs:279-316 */
            if (lwe_in[i] == 0) continue;
            size_t a_hat = (size_t)orc_modulus_switch(lwe_in[i], lgN);
            for (size_t q = 0; q < k1; q++) orc_monomial_mul_and_subtract(s->ct1 + q * N, s->ct0 + q * N, N, a_hat);
            add_external_product_f64_planes(p, f->re + i * plane, f->im + i * plane, s->ct0, s->ct1, s);
        }
    } else {
        /* deterministic order (lwe_multi_bit_programmable_bootstrapping.rs:755-800): dst = 0; dst += G (x) src */
        size_t g = p->grouping_factor, groups = n / g;
        uint64_t *src = s->ct0, *dst = s->ct1;
        for (size_t grp = 0; grp < groups && grp < max_steps; grp++) {
            prepare_multi_bit_ggsw(p, f, grp, lwe_in + grp * g, s);
            memset(dst, 0, k1 * N * 8);
            add_external_product_f64_planes(p, s->g_re, s->g_im, dst, src, s);
            uint64_t *t = src; src = dst; dst = t;
        }
        if (src != s->ct0) memcpy(s->ct0, src, k1 * N * 8);
    }
}

static void blind_rotate_f64(const orc_params *p, const orc_fourier_bsk *f, const uint64_t *lwe_in, pbs_scratch *s) {
    blind_rotate_f64_steps(p, f, lwe_in, s, (size_t)-1);
}

static void pbs_f64_with_scratch(const orc_params *p, const orc_fourier_bsk *f, const uint64_t *lwe_in,
                                 const uint64_t *acc, uint64_t *lwe_out, pbs_scratch *s) {
    size_t N = p->poly_size, k1 = p->glwe_dim + 1;
    memcpy(s->ct0, acc, k1 * N * 8);           /* bootstrap.rs:350-356 */
    blind_rotate_f64(p, f, lwe_in, s);
    orc_sample_extract0(p, s->ct0, lwe_out);   /* bootstrap.rs:358-362 */
}

/* Non-native power-of-two ciphertext modulus q = 2^log2_q (values live in the MSBs): after the blind rotation every accumulator
 * coefficient is rounded to a multiple of 2^(64 - log2_q) with SignedDecomposer(base_log = log2_q, level 1).closest_representable
 * (fft64/crypto/bootstrap.rs:318-330), then the sample is extracted (:358-362). */
void orc_pbs_f64_pow2_modulus(const orc_params *p, const orc_fourier_bsk *f, const uint64_t *lwe_in, const uint64_t *acc,
                              uint64_t *lwe_out, uint32_t log2_q) {
    size_t N = p->poly_size, k1 = p->glwe_dim + 1;
    pbs_scratch s; scratch_init(&s, p);
    memcpy(s.ct0, acc, k1 * N * 8);
    blind_rotate_f64(p, f, lwe_in, &s);
    if (log2_q < 64)
        for (size_t j = 0; j < k1 * N; j++) s.ct0[j] = orc_closest_representable(s.ct0[j], log2_q, 1);
    orc_sample_extract0(p, s.ct0, lwe_out);
    scratch_free(&s);
}

void orc_pbs_f64(const orc_params *p, const orc_fourier_bsk *f, const uint64_t *lwe_in, const uint64_t *acc, uint64_t *lwe_out) {
    pbs_scratch s; scratch_init(&s, p);
    pbs_f64_with_scratch(p, f, lwe_in, acc, lwe_out, &s);
    scratch_free(&s);
}

/* PBS that stops after n_steps blind-rotation steps (mask elements, or groups for the multi-bit PBS), then extracts the sample:
 * n_steps = 0 is LUT rotation + extraction (integer only), n_steps = 1 one external product (ggsw.rs:477-598). */
void orc_pbs_f64_partial(const orc_params *p, const orc_fourier_bsk *f, const uint64_t *lwe_in, const uint64_t *acc, uint64_t *lwe_out,
                         size_t n_steps) {
    size_t N = p->poly_size, k1 = p->glwe_dim + 1;
    pbs_scratch s; scratch_init(&s, p);
    memcpy(s.ct0, acc, k1 * N * 8);
    blind_rotate_f64_steps(p, f, lwe_in, &s, n_steps);
    orc_sample_extract0(p, s.ct0, lwe_out);
    scratch_free(&s);
}

/* Exact classic PBS: same control flow, exact integer external products (slow: O(n*N^2)). */
void orc_pbs_exact(const orc_params *p, const uint64_t *bsk_std, const uint64_t *lwe_in, const uint64_t *acc, uint64_t *lwe_out) {
    size_t N = p->poly_size, k1 = p->glwe_dim + 1, n = p->lwe_dim;
    uint32_t lgN = ilog2(N);
    size_t gl = ggsw_len(p);
    uint64_t *ct0 = (uint64_t *)malloc(k1 * N * 8), *ct1 = (uint64_t *)malloc(k1 * N * 8);
    size_t b_hat = (size_t)orc_modulus_switch(lwe_in[n], lgN);
    for (size_t q = 0; q < k1; q++) orc_monomial_div(ct0 + q * N, acc + q * N, N, b_hat);
    for (size_t i = 0; i < n; i++) {
        if (lwe_in[i] == 0) continue;
        size_t a_hat = (size_t)orc_modulus_switch(lwe_in[i], lgN);
        for (size_t q = 0; q < k1; q++) orc_monomial_mul_and_subtract(ct1 + q * N, ct0 + q * N, N, a_hat);
        orc_add_external_product_exact(p, bsk_std + i * gl, ct0, ct1);
    }
    orc_sample_extract0(p, ct0, lwe_out);
    free(ct0); free(ct1);
}

/* o += d * g in Z_2^64[X]/(X^N+1), iterating over the nonzero coefficients of g: O(N * nnz(g)), so sparse test keys are cheap */
ORC_CLONES
static void negacyclic_mul_add_by_key(uint64_t *restrict o, const uint64_t *restrict d, const uint64_t *restrict g, size_t N) {
    for (size_t b = 0; b < N; b++) {
        const uint64_t c = g[b];
        if (!c) continue;
        for (size_t a = 0; a < N - b; a++) o[a + b] += d[a] * c;
        for (size_t a = N - b; a < N; a++) o[a + b - N] -= d[a] * c;
    }
}

/* orc_add_external_product_exact with the product above and caller-owned scratch (states: k1*N, digits: N) */
static void add_external_product_exact_by_key(const orc_params *p, const uint64_t *ggsw_std, uint64_t *out, const uint64_t *glwe,
                                              uint64_t *states, uint64_t *digits) {
    size_t N = p->poly_size, k1 = p->glwe_dim + 1, L = p->pbs_level;
    uint32_t bl = p->pbs_base_log;
    uint64_t mask = ((uint64_t)1 << bl) - 1;
    for (size_t j = 0; j < k1 * N; j++)
        states[j] = orc_closest_representable(glwe[j], bl, p->pbs_level) >> (64 - bl * L);
    for (size_t lv = L; lv >= 1; lv--) {
        for (size_t row = 0; row < k1; row++) {
            for (size_t j = 0; j < N; j++) digits[j] = decompose_one_level(bl, &states[row * N + j], mask);
            for (size_t col = 0; col < k1; col++)
                negacyclic_mul_add_by_key(out + col * N, digits, ggsw_std + ((((lv - 1) * k1 + row) * k1) + col) * N, N);
        }
    }
}

/* Exact PBS, classic and multi-bit, stopping after max_steps mask elements (classic) / groups (multi-bit) like orc_pbs_f64_partial.
 * Classic: the control flow of orc_pbs_exact.  Multi-bit: the order of blind_rotate_f64_steps, with the combined GGSW
 * G = G_0 + sum_idx X^{sw_idx} * G_idx (prepare_multi_bit_ggsw) built by exact negacyclic monomial products. */
static void pbs_exact_steps_scratch(const orc_params *p, const uint64_t *bsk_std, const uint64_t *lwe_in, const uint64_t *acc,
                                    uint64_t *lwe_out, size_t max_steps, uint64_t *ct0, uint64_t *ct1, uint64_t *states,
                                    uint64_t *digits, uint64_t *G, uint64_t *mono) {
    size_t N = p->poly_size, k1 = p->glwe_dim + 1, n = p->lwe_dim, gl = ggsw_len(p);
    uint32_t lgN = ilog2(N);
    size_t b_hat = (size_t)orc_modulus_switch(lwe_in[n], lgN);
    for (size_t q = 0; q < k1; q++) orc_monomial_div(ct0 + q * N, acc + q * N, N, b_hat);
    if (p->grouping_factor == 0) {
        for (size_t i = 0; i < n && i < max_steps; i++) {
            if (lwe_in[i] == 0) continue;
            size_t a_hat = (size_t)orc_modulus_switch(lwe_in[i], lgN);
            for (size_t q = 0; q < k1; q++) orc_monomial_mul_and_subtract(ct1 + q * N, ct0 + q * N, N, a_hat);
            add_external_product_exact_by_key(p, bsk_std + i * gl, ct0, ct1, states, digits);
        }
    } else {
        size_t g = p->grouping_factor, per = (size_t)1 << g, groups = n / g;
        uint64_t *src = ct0, *dst = ct1;
        for (size_t grp = 0; grp < groups && grp < max_steps; grp++) {
            const uint64_t *base = bsk_std + grp * per * gl, *mask_elems = lwe_in + grp * g;
            memcpy(G, base, gl * 8);
            for (size_t idx = 1; idx < per; idx++) {
                uint64_t deg = 0;
                for (size_t mi = 0; mi < g; mi++) deg += (uint64_t)((idx >> (g - (mi + 1))) & 1) * mask_elems[mi];
                size_t sw = (size_t)orc_modulus_switch(deg, lgN);
                for (size_t q = 0; q < gl / N; q++) {
                    orc_monomial_mul(mono, base + idx * gl + q * N, N, sw);
                    for (size_t j = 0; j < N; j++) G[q * N + j] += mono[j];
                }
            }
            memset(dst, 0, k1 * N * 8);
            add_external_product_exact_by_key(p, G, dst, src, states, digits);
            uint64_t *t = src; src = dst; dst = t;
        }
        if (src != ct0) memcpy(ct0, src, k1 * N * 8);
    }
    orc_sample_extract0(p, ct0, lwe_out);
}

void orc_pbs_exact_steps(const orc_params *p, const uint64_t *bsk_std, const uint64_t *lwe_in, const uint64_t *acc, uint64_t *lwe_out,
                         size_t max_steps) {
    size_t N = p->poly_size, k1 = p->glwe_dim + 1, gl = ggsw_len(p);
    uint64_t *ct0 = (uint64_t *)malloc(k1 * N * 8), *ct1 = (uint64_t *)malloc(k1 * N * 8), *states = (uint64_t *)malloc(k1 * N * 8);
    uint64_t *digits = (uint64_t *)malloc(N * 8), *G = (uint64_t *)malloc(gl * 8), *mono = (uint64_t *)malloc(N * 8);
    pbs_exact_steps_scratch(p, bsk_std, lwe_in, acc, lwe_out, max_steps, ct0, ct1, states, digits, G, mono);
    free(ct0); free(ct1); free(states); free(digits); free(G); free(mono);
}

/* batch PBS without keyswitch, one ciphertext per OpenMP thread: exact (f == NULL, integer products on bsk_std) or f64 (f) */
static int pbs_batch_steps(const orc_params *p, const orc_fourier_bsk *f, const uint64_t *bsk_std, const uint64_t *luts,
                           const uint32_t *lut_idx, const uint64_t *in, uint64_t *out, size_t batch, size_t max_steps, int threads) {
    size_t big = (size_t)p->glwe_dim * p->poly_size + 1, small = p->lwe_dim + 1;
    size_t N = p->poly_size, k1 = p->glwe_dim + 1, gl = ggsw_len(p);
    (void)get_plan(N);
    int used = 1;
#ifdef _OPENMP
    if (threads <= 0) threads = omp_get_max_threads();
    used = threads;
#else
    (void)threads;
#endif
    #pragma omp parallel num_threads(threads)
    {
        pbs_scratch s; scratch_init(&s, p);
        uint64_t *states = (uint64_t *)malloc(k1 * N * 8), *digits = (uint64_t *)malloc(N * 8), *G = (uint64_t *)malloc(gl * 8);
        #pragma omp for schedule(dynamic, 1)
        for (long b = 0; b < (long)batch; b++) {
            const uint64_t *acc = luts + (size_t)(lut_idx ? lut_idx[b] : 0) * k1 * N;
            const uint64_t *x = in + (size_t)b * small;
            uint64_t *y = out + (size_t)b * big;
            if (f) {
                memcpy(s.ct0, acc, k1 * N * 8);
                blind_rotate_f64_steps(p, f, x, &s, max_steps);
                orc_sample_extract0(p, s.ct0, y);
            } else {
                pbs_exact_steps_scratch(p, bsk_std, x, acc, y, max_steps, s.ct0, s.ct1, states, digits, G, s.mono);
            }
        }
        free(states); free(digits); free(G); scratch_free(&s);
    }
    return used;
}

int orc_pbs_exact_batch(const orc_params *p, const uint64_t *bsk_std, const uint64_t *luts, const uint32_t *lut_idx,
                        const uint64_t *in, uint64_t *out, size_t batch, size_t max_steps, int threads) {
    return pbs_batch_steps(p, NULL, bsk_std, luts, lut_idx, in, out, batch, max_steps, threads);
}

int orc_pbs_f64_batch(const orc_params *p, const orc_fourier_bsk *f, const uint64_t *luts, const uint32_t *lut_idx,
                      const uint64_t *in, uint64_t *out, size_t batch, size_t max_steps, int threads) {
    return pbs_batch_steps(p, f, NULL, luts, lut_idx, in, out, batch, max_steps, threads);
}

int orc_max_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

int orc_ks_pbs_batch(const orc_params *p, const uint64_t *ksk, const orc_fourier_bsk *f,
                     const uint64_t *luts, const uint32_t *lut_idx,
                     const uint64_t *in, uint64_t *out, uint64_t *ks_out, size_t batch, int threads) {
    size_t big = (size_t)p->glwe_dim * p->poly_size + 1, small = p->lwe_dim + 1;
    size_t lut_len = (size_t)(p->glwe_dim + 1) * p->poly_size;
    (void)get_plan(p->poly_size);
    int used = 1;
#ifdef _OPENMP
    if (threads <= 0) threads = omp_get_max_threads();
    used = threads;
#else
    (void)threads;
#endif
    #pragma omp parallel num_threads(threads)
    {
        pbs_scratch s; scratch_init(&s, p);
        uint64_t *tmp = (uint64_t *)malloc(small * 8);
        #pragma omp for schedule(dynamic, 1)
        for (long b = 0; b < (long)batch; b++) {
            orc_keyswitch(p, ksk, in + (size_t)b * big, tmp);
            if (ks_out) memcpy(ks_out + (size_t)b * small, tmp, small * 8);
            const uint64_t *acc = luts + (size_t)(lut_idx ? lut_idx[b] : 0) * lut_len;
            pbs_f64_with_scratch(p, f, tmp, acc, out + (size_t)b * big, &s);
        }
        free(tmp); scratch_free(&s);
    }
    return used;
}
