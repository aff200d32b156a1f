// pbs_n512.cu -- tuned blind rotation for N = 512, k = 3, one PBS level: PARAM_MESSAGE_1_CARRY_1_KS_PBS (shortint/parameters/mod.rs:613-627),
// the first of the sets the reference benchmarks (docs/getting_started/benchmarks.md:42) that pbs_v4.cu does not serve.
//
// The generic kernel (pbs_generic.cu) runs this shape at 0.16 of the FP64 peak: one 64-thread CTA per ciphertext, radix-2 / radix-4 passes
// through one shared buffer, and every CTA pulls the whole 45 MB Fourier key through L2 on its own (3 TB/s of L2 reads at 67 k PBS/s).
// This kernel is pbs_v4.cu's data path re-cut for four polynomials of 256 complex points:
//   * 16 threads x 16 points per polynomial: the size-256 FFT is radix-16, one 16 x 16 transpose, radix-16 -- ONE exchange, and it stays
//     inside a half-warp (__syncwarp only).  A ciphertext is 64 threads = two warps, each warp two polynomials in its two halves.
//   * eight ciphertexts (16 warps, 128 registers) per SM share ONE stream of the key through a TMA-fed ring of 16 KiB pieces (a GGSW is
//     16 polynomials x 256 points = 64 KiB, as for N = 2048 / k = 1), so the key crosses L2 -> SM once per SM, not once per ciphertext.
//   * accumulator master copy and the 16 per-thread twiddles in the thread's Tensor Memory lane (tcgen05.ld / st).
//   * external product: every thread parks its 16 spectrum values in its polynomial's tile; after one barrier over the ciphertext's 64
//     threads a thread accumulates output polynomial c = its own index from the four input spectra (its own from registers).
// Same arithmetic definition as the other kernels (bootstrap.rs:242-364, ggsw.rs:477-598, fft/mod.rs:197-326).
//
// FFT: point j = T + 16 m (thread T, register m), Z_k = sum_j z_j w^j W^(jk), w = exp(i pi / 512), W = exp(-2 pi i / 256), k = k1 + 16 k2:
//   pass 1  radix-16 DIF over m of z * w^(16 m) (the pre-twist constants exp(i pi m / 32) are those of fft16_core.cuh)  -> register p1 = brev4(k1)
//   twiddle T1[p1][T] = w^T W^(T brev4(p1)) = exp(i pi T (1 - 4 brev4(p1)) / 512)
//   exchange (T, p1) -> thread T' = p1, register T       (tile rows padded to 17 elements: conflict-free both ways)
//   pass 2  radix-16 DIF over T                          -> register pv = brev4(k2)
// Thread T', register pv holds k = brev4(T') + 16 brev4(pv); the key is converted by the same device function, so the order never matters.
#include <cstdlib>

#include "kernels.h"
#include "sample_extract.cuh"
#include "pbs16_common.cuh"
#include "fft16x_slots.cuh"

namespace tb512 {
using namespace tb16k;
using namespace tb16x;

constexpr int LOGN = 9, N = 1 << LOGN, M = N / 2, K1 = 4;
constexpr int TILE = kTile256;                      // complex elements per polynomial tile (>= N u64 words for the rotated gather)
constexpr int QPP = 4;                              // frequencies (registers) per ring piece
constexpr int PIECE_CPLX = QPP * K1 * K1 * 16;      // [q 4][out poly c 4][in poly r 4][thread 16] = 1024 complex = 16 KiB
constexpr int PIECE_BYTES = PIECE_CPLX * 16;
constexpr int CHUNKS = 16 / QPP;
constexpr int NS = 5;

template <int CTS>
struct Smem {
    cplx tile[K1 * CTS][TILE];
    cplx ring[NS][PIECE_CPLX];
    unsigned long long full_bar[NS];
    unsigned int consumed[NS];
    uint32_t tmem_base;
};
static_assert(sizeof(Smem<8>) <= 227 * 1024, "shared memory budget");

// Fourier key, ring order: [ggsw i][chunk][q][out poly c][in poly r][thread 16]; register g = QPP * chunk + q
__device__ __forceinline__ size_t key_index(int i, int g, int c, int r) {
    return (((((size_t)i * CHUNKS + (g / QPP)) * QPP + (g % QPP)) * K1 + c) * K1 + r) * 16;
}

__device__ __forceinline__ uint32_t mod_switch(uint64_t x) { return (uint32_t)(((x >> (64 - LOGN - 2)) + 1) >> 1) & (2 * N - 1); }

// the 16-thread FFT over one polynomial's tile; twiddles tw[p] = T1[p][T]
struct Fft256 {
    template <class Tw>
    __device__ __forceinline__ static void fwd(double (&re)[16], double (&im)[16], cplx *tile, const Tw &twd, int T) {
        radix16_twisted_fwd(re, im);
        twd.template apply<false>(re, im);
        __syncwarp();          // the half-warp is done with the tile (rotated gather / previous exchange)
#pragma unroll
        for (int p = 0; p < 16; ++p) { cplx v; v.x = re[p]; v.y = im[p]; tile[s256_write(T, p)] = v; }
        __syncwarp();
#pragma unroll
        for (int u = 0; u < 16; ++u) { const cplx v = tile[s256_read(T, u)]; re[u] = v.x; im[u] = v.y; }
        radix16_fwd(re, im);
    }
    // inverse, scaled by 256
    template <class Tw>
    __device__ __forceinline__ static void inv(double (&re)[16], double (&im)[16], cplx *tile, const Tw &twd, int T) {
        radix16_dit_inv(re, im);
#pragma unroll
        for (int u = 0; u < 16; ++u) { cplx v; v.x = re[u]; v.y = im[u]; tile[s256_read(T, u)] = v; }
        __syncwarp();
#pragma unroll
        for (int p = 0; p < 16; ++p) { const cplx v = tile[s256_write(T, p)]; re[p] = v.x; im[p] = v.y; }
        twd.template apply<true>(re, im);
        radix16_dit_inv(re, im);
        posttwist16_inv(re, im);
    }
};

struct TmemTw {          // 16 twiddles = 64 columns of the thread's TMEM lane
    uint32_t col;
    template <bool INV>
    __device__ __forceinline__ void apply(double (&re)[16], double (&im)[16]) const {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            uint32_t v[16];
            tmem_ld16(col + 16 * k, v);
            tmem_wait_ld();
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const cplx w = cplx_from_words(v, q);
                const int p = 4 * k + q;
                const double a = re[p], b = im[p];
                if (!INV) { re[p] = DFMA(a, w.x, -DMUL(b, w.y)); im[p] = DFMA(b, w.x, DMUL(a, w.y)); }
                else { re[p] = DFMA(a, w.x, DMUL(b, w.y)); im[p] = DFMA(b, w.x, -DMUL(a, w.y)); }
            }
        }
    }
};
struct GlobalTw {
    const cplx *tbl;
    int T;
    template <bool INV>
    __device__ __forceinline__ void apply(double (&re)[16], double (&im)[16]) const {
        if (!INV) twiddle16_fwd(re, im, [&](int p) { return __ldg(tbl + p * 16 + T); });
        else twiddle16_inv(re, im, [&](int p) { return __ldg(tbl + p * 16 + T); });
    }
};

template <int CTS>
__global__ void __launch_bounds__(64 * CTS, 1)
pbs_n512_kernel(const uint64_t *__restrict__ lwe_small, const uint32_t *__restrict__ lut_idx, const uint64_t *__restrict__ luts,
                const cplx *__restrict__ bskf, const cplx *__restrict__ tbl, uint64_t *__restrict__ out,
                const uint32_t *__restrict__ out_slot, const tbk::ManyLut many, int batch, int n, int base_log, int n_iters) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int WARPS = 2 * CTS, WPQ = (WARPS + 3) / 4;        // warps that share a TMEM lane quarter
    constexpr int TW_COL = 64 * WPQ, NEED = TW_COL + 64;
    constexpr int TMEM_COLS = NEED <= 128 ? 128 : NEED <= 256 ? 256 : 512;
    Smem<CTS> &sm = *reinterpret_cast<Smem<CTS> *>(smem_raw);
    const int W = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ctl = W >> 1, r = ((W & 1) << 1) | (lane >> 4), T = lane & 15;      // ciphertext, polynomial (0..2 mask, 3 body), FFT thread
    const int ct_raw = blockIdx.x * CTS + ctl;
    const bool live = ct_raw < batch;
    const int ct = live ? ct_raw : batch - 1;
    cplx *tile = sm.tile[K1 * ctl + r];
    uint64_t *pb = reinterpret_cast<uint64_t *>(tile);
    const int ct_bar = 1 + ctl;                     // named barrier over the ciphertext's 64 threads
    const uint64_t *lwe = lwe_small + (size_t)ct * (n + 1);
    const int total_pieces = n_iters * CHUNKS;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NS; ++s) { mbar_init(&sm.full_bar[s], 1); sm.consumed[s] = 0; }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async();
    }
    if (W == 0) tmem_alloc<TMEM_COLS>(&sm.tmem_base);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t quarter = sm.tmem_base + ((uint32_t)((W & 3) * 32) << 16);
    const uint32_t tmem_mine = quarter + (uint32_t)((W >> 2) * 64);
    const TmemTw twd{quarter + (uint32_t)TW_COL};
    {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            uint32_t v[16];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const cplx t = __ldg(tbl + (4 * kk + q) * 16 + T);
                pack_cplx(t.x, t.y, v, q);
            }
            tmem_st16(twd.col + 16 * kk, v);
        }
    }
    if (threadIdx.x == 0) {
        const int first = total_pieces < NS ? total_pieces : NS;
        for (int g = 0; g < first; ++g) {
            mbar_expect_tx(&sm.full_bar[g], PIECE_BYTES);
            tma_load_1d(sm.ring[g], bskf + (size_t)g * PIECE_CPLX, PIECE_BYTES, &sm.full_bar[g]);
        }
    }

    // ---- acc <- LUT * X^(-b_hat): registers (own coefficients as u64 bit patterns), TMEM, shared -------------------------------------
    double re[16], im[16];
    {
        const uint32_t a0 = (2 * N - mod_switch(__ldg(lwe + n))) & (2 * N - 1);
        const uint64_t *lut = luts + ((size_t)(lut_idx ? lut_idx[ct] : 0) * K1 + r) * N;
#pragma unroll
        for (int m = 0; m < 16; ++m) {
            const int j = T + 16 * m;
            const uint32_t s0 = ((uint32_t)j - a0) & (2 * N - 1), s1 = ((uint32_t)(j + M) - a0) & (2 * N - 1);
            uint64_t v0 = __ldg(lut + (s0 & (N - 1))), v1 = __ldg(lut + (s1 & (N - 1)));
            v0 = s0 >= (uint32_t)N ? (uint64_t)0 - v0 : v0;
            v1 = s1 >= (uint32_t)N ? (uint64_t)0 - v1 : v1;
            pb[j] = v0; pb[j + M] = v1;
            re[m] = __longlong_as_double((long long)v0);
            im[m] = __longlong_as_double((long long)v1);
        }
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            uint32_t v[16];
#pragma unroll
            for (int mm = 0; mm < 4; ++mm) pack_cplx(re[4 * kk + mm], im[4 * kk + mm], v, mm);
            tmem_st16(tmem_mine + 16 * kk, v);
        }
        tmem_wait_st();
    }
    // the other three polynomials of the ciphertext: tile and key column of input polynomial (r + d) & 3
    const cplx *spec_d[3];
    int key_d[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const int rr = (r + d + 1) & 3;
        spec_d[d] = sm.tile[K1 * ctl + rr] + T * 17;
        key_d[d] = rr * 16;
    }

    if (CTS >= 4 && ctl >= 1 && n_iters > 0) {      // stagger the ciphertexts of an SM over an iteration
        const long long t0 = clock64(), delay = (long long)ctl * (12000 / CTS);
        while (clock64() - t0 < delay) { }
    }

    int slot = 0;
    uint32_t phase = 0;
    for (int i = 0; i < n_iters; ++i) {
        const uint32_t a = mod_switch(__ldg(lwe + i));                           // a == 0 is NOT skipped
        __syncwarp();        // the accumulator polynomial is complete in the tile (only this half-warp touches it)
#pragma unroll
        for (int m = 0; m < 16; ++m) {
            const int j = T + 16 * m;
            const uint32_t s0 = ((uint32_t)j - a) & (2 * N - 1), s1 = (s0 + M) & (2 * N - 1);
            uint64_t r0 = pb[s0 & (N - 1)], r1 = pb[s1 & (N - 1)];
            r0 = (s0 >= (uint32_t)N) ? (uint64_t)0 - r0 : r0;
            r1 = (s1 >= (uint32_t)N) ? (uint64_t)0 - r1 : r1;
            const uint64_t o0 = (uint64_t)__double_as_longlong(re[m]), o1 = (uint64_t)__double_as_longlong(im[m]);
            re[m] = (double)signed_digit_l1(r0 - o0, base_log);
            im[m] = (double)signed_digit_l1(r1 - o1, base_log);
        }
        Fft256::fwd(re, im, tile, twd, T);
        // park my spectrum in my own reader row of the tile (nobody else reads that row during the FFT)
#pragma unroll
        for (int g = 0; g < 16; ++g) { cplx v; v.x = re[g]; v.y = im[g]; tile[s256_read(T, g)] = v; }
        bar_sync(ct_bar, 64);

        // out_fft[c = r] = sum over the four input polynomials r' of F_r' * G[r'][c]
        {
            int my_slot = 0;
#pragma unroll
            for (int c = 0; c < CHUNKS; ++c) {
                if (!mbar_try_wait(&sm.full_bar[slot], phase)) mbar_wait(&sm.full_bar[slot], phase);
                const cplx *pc = sm.ring[slot] + (r * K1) * 16 + T;
#pragma unroll
                for (int q = 0; q < QPP; ++q) {
                    const int g = QPP * c + q;
                    const cplx A = pc[q * (K1 * K1 * 16) + r * 16];
                    const double fr = re[g], fi = im[g];
                    double orr = DMUL(fr, A.x);
                    orr = DFMA(-fi, A.y, orr);
                    double oi = DMUL(fr, A.y);
                    oi = DFMA(fi, A.x, oi);
#pragma unroll
                    for (int d = 0; d < 3; ++d) {
                        const cplx F = spec_d[d][g], B = pc[q * (K1 * K1 * 16) + key_d[d]];
                        orr = DFMA(F.x, B.x, orr);
                        orr = DFMA(-F.y, B.y, orr);
                        oi = DFMA(F.x, B.y, oi);
                        oi = DFMA(F.y, B.x, oi);
                    }
                    re[g] = orr; im[g] = oi;
                }
                if (lane == c) my_slot = slot;
                if (++slot == NS) { slot = 0; phase ^= 1u; }
            }
            __syncwarp();
            if (lane < CHUNKS && atomicAdd(&sm.consumed[my_slot], 1u) == WARPS - 1) {
                sm.consumed[my_slot] = 0;
                const int k2 = i * CHUNKS + lane + NS;
                if (k2 < total_pieces) {
                    __threadfence_block();
                    fence_proxy_async();
                    mbar_expect_tx(&sm.full_bar[my_slot], PIECE_BYTES);
                    tma_load_1d(sm.ring[my_slot], bskf + (size_t)k2 * PIECE_CPLX, PIECE_BYTES, &sm.full_bar[my_slot]);
                }
            }
        }
        bar_sync(ct_bar, 64);      // the other polynomials have read my spectrum: the tile is mine again

        Fft256::inv(re, im, tile, twd, T);
        __syncwarp();              // the half-warp is past its exchange reads: the tile becomes the accumulator polynomial again
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            uint32_t v[16];
            tmem_ld16(tmem_mine + 16 * kk, v);
            tmem_wait_ld();
#pragma unroll
            for (int mm = 0; mm < 4; ++mm) {
                const int m = 4 * kk + mm, j = T + 16 * m;
                uint64_t o0 = ((uint64_t)v[4 * mm + 1] << 32) | v[4 * mm];
                uint64_t o1 = ((uint64_t)v[4 * mm + 3] << 32) | v[4 * mm + 2];
                o0 += from_torus_f64(re[m]);
                o1 += from_torus_f64(im[m]);
                v[4 * mm] = (uint32_t)o0; v[4 * mm + 1] = (uint32_t)(o0 >> 32);
                v[4 * mm + 2] = (uint32_t)o1; v[4 * mm + 3] = (uint32_t)(o1 >> 32);
                pb[j] = o0; pb[j + M] = o1;
                re[m] = __longlong_as_double((long long)o0);
                im[m] = __longlong_as_double((long long)o1);
            }
            tmem_st16(tmem_mine + 16 * kk, v);
        }
        tmem_wait_st();
    }

    // sample extraction of coefficient 0 (glwe_sample_extraction.rs:91-147): mask polynomial r -> out[r N + 0] = A_r[0], out[r N + j] = -A_r[N - j]
    if (live && many.fn) {
        const int nf = tbx::many_fn_count(many, lut_idx, ct);
        tbx::extract_many_regs<16, 16, N, K1 - 1>(out, out_slot[ct], nf, tbx::many_step(many, nf, N), r, T, re, im);
    } else if (live) {
        uint64_t *o = out + (size_t)(out_slot ? out_slot[ct] : ct) * ((K1 - 1) * N + 1);
        if (r < K1 - 1) {
            uint64_t *base = o + r * N;
#pragma unroll
            for (int m = 0; m < 16; ++m) {
                const int j = T + 16 * m;
                const uint64_t v0 = (uint64_t)__double_as_longlong(re[m]), v1 = (uint64_t)__double_as_longlong(im[m]);
                if (j == 0) base[0] = v0; else base[N - j] = (uint64_t)0 - v0;
                base[N - (j + M)] = (uint64_t)0 - v1;
            }
        } else if (T == 0) {
            o[(K1 - 1) * N] = (uint64_t)__double_as_longlong(re[0]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (W == 0) tmem_dealloc<TMEM_COLS>(sm.tmem_base);
}

// std key [ggsw i][level 1][row r][col c][N] -> ring order, 16 threads per polynomial (same forward transform as the kernel)
__global__ void __launch_bounds__(32)
bsk_convert_n512_kernel(const uint64_t *__restrict__ bsk_std, cplx *__restrict__ bskf, const cplx *__restrict__ tbl, int n_polys) {
    __shared__ cplx tiles[2][TILE];
    const int T = threadIdx.x & 15, half = threadIdx.x >> 4;
    const int qd = min(2 * (int)blockIdx.x + half, n_polys - 1);      // an odd tail recomputes the last polynomial (same values, same place)
    cplx *tile = tiles[half];
    const int i = qd / (K1 * K1), r = (qd / K1) % K1, c = qd % K1;
    const uint64_t *src = bsk_std + (size_t)qd * N;
    const double scale = 2.117582368135751e-22;       // 2^-72 = 2^-64 (torus) / 256 (inverse transform)
    double re[16], im[16];
#pragma unroll
    for (int m = 0; m < 16; ++m) {
        const int j = T + 16 * m;
        re[m] = DMUL((double)(long long)src[j], scale);
        im[m] = DMUL((double)(long long)src[j + M], scale);
    }
    Fft256::fwd(re, im, tile, GlobalTw{tbl, T}, T);
#pragma unroll
    for (int g = 0; g < 16; ++g) {
        cplx v; v.x = re[g]; v.y = im[g];
        bskf[key_index(i, g, c, r) + T] = v;
    }
}

}  // namespace tb512

namespace tbk {

bool pbs_n512_supported(int poly_size, int glwe_dim, int pbs_level, int grouping_factor) {
    return poly_size == tb512::N && glwe_dim == tb512::K1 - 1 && pbs_level == 1 && grouping_factor == 0;
}

void pbs_n512_make_table(double *t) { tb16x_make_table_512(t); }

cudaError_t pbs_n512_configure() {
    cudaError_t e = cudaFuncSetAttribute(tb512::pbs_n512_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tb512::Smem<8>));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(tb512::pbs_n512_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tb512::Smem<4>));
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(tb512::pbs_n512_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tb512::Smem<1>));
}

cudaError_t launch_pbs_n512(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskf, const void *tbl,
                            uint64_t *out, const uint32_t *out_slot, tbk::ManyLut many, int batch, int n, int base_log, int n_iters, cudaStream_t stream) {
    if (batch <= 0) return cudaSuccess;
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const tb::cplx *bk = reinterpret_cast<const tb::cplx *>(bskf), *tb = reinterpret_cast<const tb::cplx *>(tbl);
    if (batch <= sms)
        tb512::pbs_n512_kernel<1><<<batch, 64, sizeof(tb512::Smem<1>), stream>>>(lwe_small, lut_idx, luts, bk, tb, out, out_slot, many, batch, n, base_log, n_iters);
    else if (batch <= 4 * sms)
        tb512::pbs_n512_kernel<4><<<(batch + 3) / 4, 256, sizeof(tb512::Smem<4>), stream>>>(lwe_small, lut_idx, luts, bk, tb, out, out_slot, many, batch, n, base_log, n_iters);
    else
        tb512::pbs_n512_kernel<8><<<(batch + 7) / 8, 512, sizeof(tb512::Smem<8>), stream>>>(lwe_small, lut_idx, luts, bk, tb, out, out_slot, many, batch, n, base_log, n_iters);
    return cudaGetLastError();
}

cudaError_t launch_bsk_convert_n512(const uint64_t *bsk_std, void *bskf, const void *tbl, int n_polys, cudaStream_t stream) {
    tb512::bsk_convert_n512_kernel<<<(n_polys + 1) / 2, 32, 0, stream>>>(bsk_std, reinterpret_cast<tb::cplx *>(bskf), reinterpret_cast<const tb::cplx *>(tbl), n_polys);
    return cudaGetLastError();
}

}  // namespace tbk
