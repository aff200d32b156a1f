// leveled.cu -- batched leveled (PBS-free) shortint operations on an arena of LWE ciphertexts.
//
// Replaces the element-wise u64 wrapping loops of
//   shortint/server_key/add.rs:520-524        unchecked_add_assign     (lwe_linear_algebra.rs:68)
//   shortint/server_key/scalar_mul.rs:520-536 unchecked_scalar_mul_assign
//   shortint/server_key/scalar_add.rs:211-218 unchecked_scalar_add_assign (plaintext add on the body)
//   core_crypto/algorithms/lwe_linear_algebra.rs:703,384 lwe_ciphertext_sub_assign / plaintext_sub_assign
//   integer/server_key/radix_parallel/scalar_comparison.rs:104-139 pack_block_chunk (hi * msg_mod + lo)
//   shortint/server_key/mod.rs:684-721        create_trivial (no terms, body only)
// One instruction = one output ciphertext = sum_k coef_k * in_k (+ plaintext on the body word); the host
// composes chains of leveled ops into a single instruction, so a tree level needs one launch.
// HBM-bound: (terms + 1) * 16 392 bytes per instruction, coalesced 8-byte accesses.
#include "kernels.h"

namespace tblin {

__global__ void __launch_bounds__(256)
linear_kernel(uint64_t *__restrict__ arena, const tbk::LinInstr *__restrict__ instrs, const tbk::LinTerm *__restrict__ terms,
              int n_instrs, int lwe_len) {
    const int i = blockIdx.x;
    if (i >= n_instrs) return;
    const tbk::LinInstr ins = instrs[i];
    uint64_t *out = arena + (size_t)ins.out_slot * lwe_len;
    for (int j = threadIdx.x; j < lwe_len; j += blockDim.x) {
        uint64_t acc = (j == lwe_len - 1) ? ins.body_add : 0;
        for (uint32_t t = ins.term_begin; t < ins.term_end; ++t) {
            const tbk::LinTerm tm = terms[t];
            acc += (uint64_t)tm.coef * arena[(size_t)tm.slot * lwe_len + j];
        }
        out[j] = acc;
    }
}

}  // namespace tblin

namespace tblin {
// dst row o = arena row slots[o] (the outputs of a program, gathered so that they leave the device in ONE copy)
__global__ void __launch_bounds__(256) gather_rows_kernel(const uint64_t *__restrict__ arena, const uint32_t *__restrict__ slots,
                                                          uint64_t *__restrict__ dst, int lwe_len) {
    const uint64_t *src = arena + (size_t)slots[blockIdx.x] * lwe_len;
    uint64_t *d = dst + (size_t)blockIdx.x * lwe_len;
    for (int j = threadIdx.x; j < lwe_len; j += blockDim.x) d[j] = src[j];
}
}  // namespace tblin

namespace tblin {
// Non-native power-of-two ciphertext modulus 2^log2_q (bootstrap.rs:318-330): the reference rounds every accumulator coefficient with
// SignedDecomposer(log2_q, 1).closest_representable BEFORE the sample extraction.  Applied to the extracted sample instead: the words
// that sample extraction negated (glwe_sample_extraction.rs:91-147: every mask word except the first of each polynomial) are rounded as
// -round(-x), the others as round(x), which is the same value bit for bit, ties included.
// A many-LUT row of function f (kernels.h ManyLut) was extracted at monomial t_f: there the negated words are the mask words past t_f of
// each polynomial.
__global__ void __launch_bounds__(256) round_pow2_kernel(uint64_t *__restrict__ out, const uint32_t *__restrict__ out_slot,
                                                         const uint32_t *__restrict__ lut_idx, const tbk::ManyLut many, int poly_size,
                                                         int lwe_len, int log2_q) {
    const int nf = many.fn ? (int)many.fn[lut_idx ? lut_idx[blockIdx.x] : 0] : 1;
    const int step = many.fn ? (many.total / nf) * (poly_size / many.total) : 0;
    const int shift = 64 - log2_q - 1;
    for (int f = 0; f < nf; ++f) {
        uint64_t *row = out + ((size_t)(out_slot ? out_slot[blockIdx.x] : blockIdx.x) + f) * lwe_len;
        const int t = f * step;
        for (int j = threadIdx.x; j < lwe_len; j += blockDim.x) {
            const bool negated = j != lwe_len - 1 && (j % poly_size) > t;
            uint64_t x = row[j];
            if (negated) x = (uint64_t)0 - x;
            x = (((x >> shift) + 1) & ~(uint64_t)1) << shift;
            row[j] = negated ? (uint64_t)0 - x : x;
        }
    }
}

__global__ void __launch_bounds__(256) iota_rows_kernel(uint32_t *__restrict__ rows, size_t n, uint32_t stride) {
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i < n) rows[i] = (uint32_t)(i * stride);
}
}  // namespace tblin

namespace tbk {

cudaError_t launch_round_pow2(uint64_t *out, const uint32_t *out_slot, const uint32_t *lut_idx, ManyLut many, int batch, int poly_size,
                              int lwe_len, int log2_q, cudaStream_t stream) {
    if (batch <= 0 || log2_q >= 64) return cudaSuccess;
    tblin::round_pow2_kernel<<<batch, 256, 0, stream>>>(out, out_slot, lut_idx, many, poly_size, lwe_len, log2_q);
    return cudaGetLastError();
}

cudaError_t launch_iota_rows(uint32_t *rows, size_t n, uint32_t stride, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    tblin::iota_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(rows, n, stride);
    return cudaGetLastError();
}

cudaError_t launch_gather_rows(const uint64_t *arena, const uint32_t *slots, uint64_t *dst, int n_rows, int lwe_len, cudaStream_t stream) {
    if (n_rows <= 0) return cudaSuccess;
    tblin::gather_rows_kernel<<<n_rows, 256, 0, stream>>>(arena, slots, dst, lwe_len);
    return cudaGetLastError();
}

cudaError_t launch_linear(uint64_t *arena, const LinInstr *instrs, const LinTerm *terms, int n_instrs, int lwe_len,
                          cudaStream_t stream) {
    if (n_instrs <= 0) return cudaSuccess;
    tblin::linear_kernel<<<n_instrs, 256, 0, stream>>>(arena, instrs, terms, n_instrs, lwe_len);
    return cudaGetLastError();
}

}  // namespace tbk
