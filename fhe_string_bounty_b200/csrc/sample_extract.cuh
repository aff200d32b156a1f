// sample_extract.cuh -- the many-LUT epilogue shared by the PBS kernels (tfhe-rs extract_lwe_sample_from_glwe_ciphertext at monomial t,
// glwe_sample_extraction.rs:91-147): mask word q of polynomial r is A_r[t - q] for q <= t and -A_r[N + t - q] otherwise; the body is B[t].
// Function f of a many-LUT accumulator (kernels.h ManyLut) is extracted at t_f = f * (total / F) * (N / total).
#pragma once
#include <cstdint>

#include "kernels.h"

namespace tbx {

__device__ __forceinline__ int many_fn_count(const tbk::ManyLut &many, const uint32_t *lut_idx, int ct) {
    return (int)many.fn[lut_idx ? lut_idx[ct] : 0];
}

__device__ __forceinline__ int many_step(const tbk::ManyLut &many, int nf, int N) { return (many.total / nf) * (N / many.total); }

// coefficient j of a mask polynomial (row base `o_r`) extracted at monomial t
__device__ __forceinline__ void extract_coeff_at(uint64_t *o_r, int N, int t, int j, uint64_t v) {
    const int d = t - j;
    if (d >= 0) o_r[d] = v; else o_r[N + d] = (uint64_t)0 - v;
}

// The register-resident kernels: this thread holds coefficients j = T + STRIDE * m (re[m]) and j + N / 2 (im[m]) of polynomial r as u64
// bit patterns; polynomials 0 ... K - 1 are the mask, K the body.  Rows out + (row0 + f) * (K * N + 1), f < nf.
template <int REGS, int STRIDE, int N, int K>
__device__ __forceinline__ void extract_many_regs(uint64_t *out, size_t row0, int nf, int step, int r, int T, const double (&re)[REGS],
                                                  const double (&im)[REGS]) {
    for (int f = 0; f < nf; ++f) {
        const int t = f * step;
        uint64_t *o = out + (row0 + f) * ((size_t)K * N + 1);
        if (r < K) {
#pragma unroll
            for (int m = 0; m < REGS; ++m) {
                const int j = T + STRIDE * m;
                extract_coeff_at(o + (size_t)r * N, N, t, j, (uint64_t)__double_as_longlong(re[m]));
                extract_coeff_at(o + (size_t)r * N, N, t, j + N / 2, (uint64_t)__double_as_longlong(im[m]));
            }
        } else {
#pragma unroll
            for (int m = 0; m < REGS; ++m) {
                const int j = T + STRIDE * m;
                if (j == t) o[(size_t)K * N] = (uint64_t)__double_as_longlong(re[m]);
                if (j + N / 2 == t) o[(size_t)K * N] = (uint64_t)__double_as_longlong(im[m]);
            }
        }
    }
}

// The shared- / global-memory accumulator kernels: acc = [K + 1][N], `threads` threads starting at t0
__device__ __forceinline__ void extract_many_acc(uint64_t *out, size_t row0, int nf, int step, const uint64_t *acc, int N, int K, int t0,
                                                 int threads) {
    const size_t len = (size_t)K * N + 1;
    for (int f = 0; f < nf; ++f) {
        const int t = f * step;
        uint64_t *dst = out + (row0 + f) * len;
        for (int r = 0; r < K; ++r)
            for (int q = t0; q < N; q += threads) dst[r * N + q] = q <= t ? acc[r * N + t - q] : (uint64_t)0 - acc[r * N + N + t - q];
        if (t0 == 0) dst[(size_t)K * N] = acc[(size_t)K * N + t];
    }
}

}  // namespace tbx
