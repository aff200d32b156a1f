// kernels.h -- internal launcher interface between the C-ABI layer (c_api.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

namespace tbk {

// Many-LUT PBS (tfhe-rs generate_many_lookup_table / apply_many_lookup_table): the accumulator of lookup table l stacks fn[l] functions,
// function f in boxes [f * chunk, (f + 1) * chunk) with chunk = total / fn[l] (total = msg_mod * carry_mod), and the PBS epilogue extracts
// function f at monomial f * chunk * (N / total) into row out_slot[ct] + f.  fn == nullptr: one function per table, extracted at monomial 0
// into row out_slot[ct] (the single-function epilogue, unchanged).
struct ManyLut {
    const uint32_t *fn = nullptr;   // per lookup table: its function count F (1 ... total)
    int total = 0;
};

// keyswitch.cu
int ks_padded_cols(int n);
int ks_max_level();          // the largest level count whose two pipeline stages fit in 227 KB of shared memory
cudaError_t ks_configure();
cudaError_t launch_ksk_pack(const uint64_t *ksk, uint64_t *packed, uint64_t *colsum, int rows, int n, cudaStream_t stream);
cudaError_t launch_keyswitch(const uint64_t *lwe_in, const uint32_t *in_slot, const uint64_t *ksk_packed, const uint64_t *colsum, uint64_t *lwe_out,
                             int batch, int in_dim, int n, int base_log, int level, cudaStream_t stream);

// keyswitch_mma.cu
bool ks_mma_supported(int level);
cudaError_t launch_ksk_planes(const uint64_t *packed, uint8_t *bmat, int rows, int ldk, cudaStream_t stream);
cudaError_t launch_keyswitch_mma(const uint64_t *lwe_in, const uint32_t *in_slot, uint8_t *digits_scratch, const uint8_t *bmat,
                                 const uint64_t *colsum, uint64_t *lwe_out, int batch, int in_dim, int n, int base_log, int level,
                                 int ms_log2_2n, cudaStream_t stream);
size_t ks_mma_digits_bytes(int batch, int in_dim, int level);
cudaError_t launch_ks_digits(const uint64_t *lwe_in, const uint32_t *in_slot, uint8_t *digits, int batch, int batch_pad, int in_dim,
                             int base_log, int level, cudaStream_t stream);

// keyswitch_tc.cu: the same GEMM on tcgen05.mma kind::i8 (TMA operands, accumulator in Tensor Memory); same digit matrix and key planes
bool ks_tc_supported(int in_dim, int level);
size_t ks_tc_digits_bytes(int batch, int in_dim, int level);
cudaError_t launch_keyswitch_tc(const uint64_t *lwe_in, const uint32_t *in_slot, uint8_t *digits_scratch, const uint8_t *bmat,
                                const uint64_t *colsum, uint64_t *lwe_out, int batch, int in_dim, int n, int base_log, int level,
                                int ms_log2_2n, cudaStream_t stream);

// pbs_v4.cu (tbl16 = the two twiddle tables of fft16_core.cuh, 1024 + 64 complex values)
cudaError_t pbs_v4_configure();
cudaError_t launch_pbs_classic_v4(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskf4,
                                  const void *tbl16, uint64_t *out, const uint32_t *out_slot, ManyLut many, int batch, int n, int base_log,
                                  int n_iters, int small_is_u16, int cts, cudaStream_t stream);
cudaError_t launch_bsk_convert_v4(const uint64_t *bsk_std, void *bskf4, const void *tbl16, int n_polys, cudaStream_t stream);
// probe.cu
cudaError_t launch_fp64_peak(double *sink, int blocks, int iters, cudaStream_t stream);

// leveled.cu
struct LinInstr {          // out = sum_k coef[k] * in[k]  (+ body_add on the body word); terms in [term_begin, term_end)
    uint32_t out_slot, term_begin, term_end, pad;
    uint64_t body_add;
};
struct LinTerm {
    uint32_t slot, pad;
    int64_t coef;
};
cudaError_t launch_linear(uint64_t *arena, const LinInstr *instrs, const LinTerm *terms, int n_instrs, int lwe_len,
                          cudaStream_t stream);

// pbs_v8.cu: the narrow-level (batch <= 2 * SM count) instance, 8 FFT points per thread; tbl8 = fft8_core.cuh tables (24 x 128 complex)
cudaError_t pbs_v8_configure();
cudaError_t launch_pbs_classic_v8(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskf8,
                                  const void *tbl8, uint64_t *out, const uint32_t *out_slot, ManyLut many, int batch, int n, int base_log,
                                  int n_iters, int small_is_u16, int cluster_max /* levels of at most this many ciphertexts: one per 2-SM cluster */,
                                  cudaStream_t stream);
cudaError_t launch_bsk_convert_v8(const uint64_t *bsk_std, void *bskf8, const void *tbl8, int n_polys, cudaStream_t stream);
// pbs_multibit_v4.cu (16 FFT points per thread, 1/2/4 ciphertexts per CTA; tbl16 = fft16_core.cuh tables)
cudaError_t pbs_multibit_v4_configure();
cudaError_t launch_pbs_multibit_v4(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskm,
                                   const void *tbl16, const void *roots, uint64_t *out, const uint32_t *out_slot, ManyLut many, int batch, int n,
                                   int base_log, int n_groups, cudaStream_t stream);
cudaError_t launch_bsk_convert_multibit_v4(const uint64_t *bsk_std, void *bskm, const void *tbl16, int n_polys, cudaStream_t stream);

// pbs_multibit_v8.cu: multi-bit narrow levels (batch <= SM count), 8 FFT points per thread, one ciphertext per CTA
cudaError_t pbs_multibit_v8_configure();
cudaError_t launch_pbs_multibit_v8(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskm8,
                                   const void *tbl8, const void *roots, uint64_t *out, const uint32_t *out_slot, ManyLut many, int batch, int n,
                                   int base_log, int n_groups, int cluster_max, cudaStream_t stream);
cudaError_t launch_bsk_convert_multibit_v8(const uint64_t *bsk_std, void *bskm8, const void *tbl8, int n_polys, cudaStream_t stream);

// pbs_generic.cu: classic PBS for any (poly_size <= 8192, glwe_dim, pbs_level) of shortint/parameters/mod.rs; tw = exp(i*pi*j/N), j < N/2
bool pbs_generic_supported(int poly_size, int glwe_dim);
cudaError_t launch_pbs_generic(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskf, const void *tw,
                               uint64_t *out, const uint32_t *out_slot, ManyLut many, int batch, int n, int poly_size, int glwe_dim, int base_log,
                               int levels, int grouping_factor /* 0 = classic, 2 / 3 = multi-bit (poly_size <= 8192) */, int n_iters,
                               cudaStream_t stream);
cudaError_t launch_bsk_convert_generic(const uint64_t *bsk_std, void *bskf, const void *tw, size_t n_polys, int poly_size, cudaStream_t stream);

// pbs_n512.cu: tuned blind rotation for N = 512, k = 3, one level (PARAM_MESSAGE_1_CARRY_1_KS_PBS); tbl = 256 complex twiddles
bool pbs_n512_supported(int poly_size, int glwe_dim, int pbs_level, int grouping_factor);
void pbs_n512_make_table(double *t /* 512 doubles */);
cudaError_t pbs_n512_configure();
cudaError_t launch_pbs_n512(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskf, const void *tbl,
                            uint64_t *out, const uint32_t *out_slot, ManyLut many, int batch, int n, int base_log, int n_iters, cudaStream_t stream);
cudaError_t launch_bsk_convert_n512(const uint64_t *bsk_std, void *bskf, const void *tbl, int n_polys, cudaStream_t stream);

// pbs_n8192.cu: tuned blind rotation for N = 8192, k = 1, two levels (PARAM_MESSAGE_3_CARRY_3_KS_PBS and siblings): one ciphertext per
// two-SM cluster; tbl = 4096 + 256 complex twiddles
bool pbs_n8192_supported(int poly_size, int glwe_dim, int pbs_level, int pbs_base_log, int grouping_factor);
void pbs_n8192_make_table(double *t /* 2 * 4352 doubles */);
cudaError_t pbs_n8192_configure();
cudaError_t launch_pbs_n8192(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskf, const void *tbl,
                             uint64_t *out, const uint32_t *out_slot, ManyLut many, int batch, int n, int base_log, int n_iters, int n_ggsw,
                             cudaStream_t stream);
cudaError_t launch_bsk_convert_n8192(const uint64_t *bsk_std, void *bskf, const void *tbl, int n_ggsw, cudaStream_t stream);

// leveled.cu: rounding of PBS outputs to a non-native power-of-two ciphertext modulus (bootstrap.rs:318-330)
cudaError_t launch_round_pow2(uint64_t *out, const uint32_t *out_slot, const uint32_t *lut_idx, ManyLut many, int batch, int poly_size, int lwe_len, int log2_q, cudaStream_t stream);
cudaError_t launch_iota_rows(uint32_t *rows, size_t n, uint32_t stride, cudaStream_t stream);   // rows[i] = i * stride
cudaError_t launch_gather_rows(const uint64_t *arena, const uint32_t *slots, uint64_t *dst, int n_rows, int lwe_len, cudaStream_t stream);

// seeded.cu: dst row g = [mask_len words of the AES-128 CTR stream of `seed` | body_len words copied from bodies]
cudaError_t launch_seeded_expand(const uint8_t seed[16], uint64_t *dst, const uint64_t *bodies, size_t n_rows, uint32_t mask_len,
                                 uint32_t body_len, cudaStream_t stream);
}  // namespace tbk
