// pbs_v4.cu -- blind rotation for wide levels: the Fourier key streamed once per SM through a TMA-fed shared-memory ring, the
// accumulator's master copy in Tensor Memory, 16 FFT points per thread (fft16_core.cuh): four warps per ciphertext, lanes 0-15 of a
// warp on the mask polynomial and lanes 16-31 on the body polynomial, four ciphertexts (16 warps) per SM.
//
// Same arithmetic definition as the reference (bootstrap.rs:242-364, ggsw.rs:477-598, fft/mod.rs:197-326); the FFT evaluates the same
// 1024 frequencies as concrete-fft, only the butterfly order (hence FP64 rounding) differs.
//
// What bounds the kernel (ncu, scripts/microbench/pipes.cu and fp64.cu, profiles/r02_*): every variant tried in round 2 -- four or
// five ciphertexts per SM, spectrum exchange through shared memory or through shuffles, exchange A through shared memory or through
// Tensor Memory -- ends at the same 0.52-0.56 instructions per cycle and scheduler, i.e. the run time follows the INSTRUCTION COUNT
// (2.65 k per warp and iteration, half of them FP64 at two dispatch cycles each), not the shared-memory pipe (46-76 % busy) and not the
// FP64 pipe (44-55 %).  Measured pipe costs: LDS.128 4.25, STS.128 4.73, SHFL 2.4 cycles per warp instruction on ONE shared pipe;
// tcgen05.ld / st 11.3 / 6.9 cycles per 2 KiB on a separate, concurrent path.  Tried and dropped: a fifth ciphertext per SM (96
// registers: +9 % time), exchange A through Tensor Memory with a ciphertext's four warps in one lane quarter (shared-memory pipe 76 ->
// 47 %, but +31 % instructions for uniform-register address moves, warp-part twiddles and spills: +34 % time).  Kept: the two
// polynomials of a ciphertext in the two halves of each warp, so that the spectrum exchange of the external product is a lane ^ 16
// shuffle (two barriers and 32 shared-memory instructions per thread and iteration fewer).  The rotated gather takes its byte offset
// and wrap mask as shifts of one index and its digit from the high word of one three-input add (fft_core.cuh rot_gather /
// rot_sub_digit): the main loop of the 4-per-SM instance went from 2 815 to 2 623 instructions, 98.2 -> 95.0 ms per 8192 (B200).
// Shared memory per 4-ciphertext CTA: 8 x 17 KiB polynomial tiles (rotated-gather source, then exchange tile) + 5 x 16 KiB ring.
// TMEM: 64 columns per ciphertext (accumulator master copy) + 80 columns of per-thread FFT twiddles.
// Named barriers: one per ciphertext (128 threads).
#include <cstdlib>

#include "kernels.h"
#include "pbs16_common.cuh"

namespace tb4 {
using namespace tb16k;

constexpr int QPP = 4;                 // frequencies (registers) per ring piece
constexpr int PIECE_CPLX = 2 * 2 * QPP * 64;   // one chunk: [out poly 2][sel 2][q QPP][thread 64] = 16 KiB
constexpr int PIECE_BYTES = PIECE_CPLX * 16;
constexpr int CHUNKS_PER_ITER = 16 / QPP;
template <int CTS> struct RingSlots { static constexpr int value = CTS == 3 ? 7 : 5; };   // 80 KiB = 1.25 iterations of key (112 KiB beside three ciphertexts)

template <int CTS>
struct Smem {
    static constexpr int NS = RingSlots<CTS>::value;
    cplx tile[2 * CTS][kTileCplx];     // 17 KiB per polynomial
    cplx ring[NS][PIECE_CPLX];
    unsigned long long full_bar[NS];
    unsigned int consumed[NS];
    uint32_t tmem_base;
};
static_assert(sizeof(Smem<4>) <= 227 * 1024, "shared memory budget");

// Fourier key, v4 layout: [ggsw i][chunk 16/QPP][out poly c][sel: 0 = row c, 1 = row 1-c][q QPP][thread 64]; register g = QPP*chunk + q
// (QPP = 4 measured 101.9 ms per 8192 against 104.1 ms for QPP = 2; QPP = 8 leaves too few slots for the ciphertexts' stagger)
__device__ __forceinline__ size_t bskf4_index(int i, int chunk, int c, int sel, int q) {
    return ((((size_t)(i * CHUNKS_PER_ITER + chunk) * 2 + c) * 2 + sel) * QPP + q) * 64;
}
// piece k = i * CHUNKS_PER_ITER + chunk: 16 KiB, contiguous in the layout above
__device__ __forceinline__ const cplx *piece_src(const cplx *bskf4, int k) { return bskf4 + (size_t)k * PIECE_CPLX; }

template <int CTS>
__global__ void __launch_bounds__(128 * CTS, 1)
pbs_classic_kernel_v4(const uint64_t *__restrict__ lwe_small, const uint32_t *__restrict__ lut_idx, const uint64_t *__restrict__ luts,
                      const cplx *__restrict__ bskf4, const cplx *__restrict__ tbl16, uint64_t *__restrict__ out,
                      const uint32_t *__restrict__ out_slot, int batch, int n, int base_log, int n_iters, int small_is_u16) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int TMEM_COLS = CTS >= 3 ? 512 : 256, CONSUMERS = 4 * CTS;   // every warp reads every ring piece
    constexpr int NS = Smem<CTS>::NS;
    constexpr int TW_COL = 64 * CTS;                                        // per-thread twiddles after the accumulators
    Smem<CTS> &sm = *reinterpret_cast<Smem<CTS> *>(smem_raw);
    const int W = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // warp -> (ciphertext, quarter of the FFT threads); HALF-warp -> polynomial: lanes 0-15 work on the mask polynomial, lanes 16-31 on
    // the body polynomial, both as the FFT threads T = 16 k + (lane & 15).  Lane l and lane l ^ 16 hold the two polynomials' spectra
    // at the SAME frequencies.  Every scheduler (warp id % 4) hosts one warp of each ciphertext; the ciphertexts are started a fraction
    // of an iteration apart (stagger below).
    const int ctl = W >> 2, k = W & 3;
    const int w = lane >> 4, T = (k << 4) | (lane & 15), P = 2 * ctl + w;
    const int ct_raw = blockIdx.x * CTS + ctl;
    const bool live = ct_raw < batch;
    const int ct = live ? ct_raw : batch - 1;        // ragged tail: recompute the last ciphertext, skip the store
    cplx *tile = sm.tile[P];
    uint64_t *pb = reinterpret_cast<uint64_t *>(tile);   // the polynomial (2048 words) for the rotated gather
    const CtSync ct_sync{1 + ctl};        // exchange A crosses the ciphertext's four warps (both polynomials travel together)
    const uint64_t *lwe = lwe_small + (size_t)ct * (n + 1);
    const uint16_t *lwe16 = reinterpret_cast<const uint16_t *>(lwe_small) + (size_t)ct * (n + 1);
    const int total_pieces = n_iters * CHUNKS_PER_ITER;

    // ---- one-time setup: twiddle tables, barriers, TMEM, first ring fill ---------------------------------------------------
    if (threadIdx.x == 0) {
        for (int s = 0; s < NS; ++s) { mbar_init(&sm.full_bar[s], 1); sm.consumed[s] = 0; }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async();
    }
    if (W == 0) tmem_alloc<TMEM_COLS>(&sm.tmem_base);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t quarter = sm.tmem_base + ((uint32_t)((W & 3) * 32) << 16);       // lane quarter = warp id % 4
    const uint32_t tmem_mine = quarter + (uint32_t)(ctl * 64);                      // this warp's accumulator columns
    const TmemTwiddles twd{quarter + (uint32_t)TW_COL};
    {   // this thread's twiddles -> TMEM (5 x 16 columns: T1[p][T], p = 0..15, then the three pass-2 twiddles)
#pragma unroll
        for (int kk = 0; kk < 5; ++kk) {
            uint32_t v[16];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const cplx t = kk < 4 ? __ldg(tbl16 + (4 * kk + q) * 64 + T) : __ldg(tbl16 + kM + 16 * (q < 3 ? q : 0) + (T & 15));
                pack_cplx(t.x, t.y, v, q);
            }
            tmem_st16(twd.col + 16 * kk, v);
        }
    }
    if (threadIdx.x == 0) {
        const int first = total_pieces < NS ? total_pieces : NS;
        for (int g = 0; g < first; ++g) {
            mbar_expect_tx(&sm.full_bar[g], PIECE_BYTES);
            tma_load_1d(sm.ring[g], piece_src(bskf4, g), PIECE_BYTES, &sm.full_bar[g]);
        }
    }

    // ---- acc <- LUT * X^(-b_hat): registers (own coefficients as u64 bit patterns in re/im), TMEM, shared ------------------------
    double re[16], im[16];
    {
        const uint32_t b_hat = (small_is_u16 ? (uint32_t)__ldg(lwe16 + n) : modulus_switch_2n(__ldg(lwe + n))) & (2 * kN - 1);
        const uint32_t a0 = (2 * kN - b_hat) & (2 * kN - 1);
        const uint64_t *lut = luts + ((size_t)(lut_idx ? lut_idx[ct] : 0) * 2 + w) * kN;
#pragma unroll
        for (int m = 0; m < 16; ++m) {
            const int j = T + 64 * m;
            int s0, s1; bool n0, n1;
            rot_src(j, a0, s0, n0);
            rot_src(j + kM, a0, s1, n1);
            uint64_t v0 = __ldg(lut + s0), v1 = __ldg(lut + s1);
            v0 = n0 ? (uint64_t)0 - v0 : v0;
            v1 = n1 ? (uint64_t)0 - v1 : v1;
            pb[j] = v0; pb[j + kM] = v1;
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

    // stagger: ciphertext c starts c / CTS of an iteration after ciphertext 0, so that the FP64-heavy and the shared-memory-heavy phases
    // of the ciphertexts do not coincide (a clock-based delay measured the same as a barrier hand-shake)
    if (CTS >= 3 && ctl >= 1 && n_iters > 0) {
        const long long t0 = clock64(), delay = (long long)ctl * (20000 / CTS);
        while (clock64() - t0 < delay) { }
    }

    int slot = 0;            // ring position (0 .. NS-1) of this iteration's first piece
    uint32_t phase = 0;

    for (int i = 0; i < n_iters; ++i) {
        const uint32_t a = (small_is_u16 ? (uint32_t)__ldg(lwe16 + i) : modulus_switch_2n(__ldg(lwe + i))) & (2 * kN - 1);   // a == 0 is NOT skipped
        ct_sync();      // the accumulator polynomial is complete in shared memory

        // ct1 = acc * X^a - acc, level-1 signed digit, folded (own coefficients come from the registers)
#pragma unroll
        for (int m = 0; m < 16; ++m) {
            const int j = T + 64 * m;
            const uint64_t o0 = (uint64_t)__double_as_longlong(re[m]), o1 = (uint64_t)__double_as_longlong(im[m]);
            const uint32_t u = ((uint32_t)j - a) << (31 - kLogN);
            uint32_t wrap0, wrap1;
            const uint64_t r0 = rot_gather(pb, u, wrap0), r1 = rot_gather(pb, u + ((uint32_t)kM << (31 - kLogN)), wrap1);
            re[m] = (double)rot_sub_digit(r0, wrap0, o0, base_log);
            im[m] = (double)rot_sub_digit(r1, wrap1, o1, base_log);
        }
        fft16_fwd(re, im, tile, twd, T, ct_sync);    // its first barrier also ends the rotated gather: nobody writes the tile before it

        // out_fft[w] = F_w * G[w][w] + F_{1-w} * G[1-w][w], GGSW pieces from the ring, the other polynomial's spectrum from lane ^ 16.
        // Nothing is synchronised inside the loop (the compiler is free to run chunk c+1's loads under chunk c's arithmetic); after it
        // lane c counts this warp out of piece c's slot, and the last of the 4 * CTS warps to leave a slot re-arms it with the piece NS
        // chunks ahead (measured against releasing each slot right after its chunk: 104.7 vs 106.0 ms per 8192).
        {
            int my_slot = 0;
#pragma unroll
            for (int c = 0; c < CHUNKS_PER_ITER; ++c) {
                if (!mbar_try_wait(&sm.full_bar[slot], phase)) mbar_wait(&sm.full_bar[slot], phase);
                const cplx *pc = sm.ring[slot] + (w * 2) * QPP * 64 + T;
#pragma unroll
                for (int q = 0; q < QPP; ++q) {
                    const int g = QPP * c + q;
                    const cplx A = pc[q * 64], B = pc[(QPP + q) * 64];
                    const double fr = re[g], fi = im[g];
                    cplx F;       // the other polynomial's spectrum at this frequency: lane ^ 16
                    F.x = __shfl_xor_sync(0xffffffffu, fr, 16);
                    F.y = __shfl_xor_sync(0xffffffffu, fi, 16);
                    double orr = DMUL(fr, A.x);
                    orr = DFMA(-fi, A.y, orr);
                    orr = DFMA(F.x, B.x, orr);
                    orr = DFMA(-F.y, B.y, orr);
                    double oi = DMUL(fr, A.y);
                    oi = DFMA(fi, A.x, oi);
                    oi = DFMA(F.x, B.y, oi);
                    oi = DFMA(F.y, B.x, oi);
                    re[g] = orr; im[g] = oi;
                }
                if (lane == c) my_slot = slot;
                if (++slot == NS) { slot = 0; phase ^= 1u; }
            }
            __syncwarp();     // every lane's loads from the ring have returned (their values fed the arithmetic above)
            if (lane < CHUNKS_PER_ITER && atomicAdd(&sm.consumed[my_slot], 1u) == CONSUMERS - 1) {
                sm.consumed[my_slot] = 0;
                const int k2 = i * CHUNKS_PER_ITER + lane + NS;
                if (k2 < total_pieces) {
                    __threadfence_block();
                    fence_proxy_async();
                    mbar_expect_tx(&sm.full_bar[my_slot], PIECE_BYTES);
                    tma_load_1d(sm.ring[my_slot], piece_src(bskf4, k2), PIECE_BYTES, &sm.full_bar[my_slot]);
                }
            }
        }

        fft16_inv(re, im, tile, twd, T, ct_sync);
        ct_sync();      // everyone is past its exchange-B reads: the tile becomes the accumulator polynomial again

        // acc += from_torus(.): master copy in TMEM, new values to registers (next gather's "own") and shared (next rotation)
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            uint32_t v[16];
            tmem_ld16(tmem_mine + 16 * kk, v);
            tmem_wait_ld();
#pragma unroll
            for (int mm = 0; mm < 4; ++mm) {
                const int m = 4 * kk + mm, j = T + 64 * m;
                uint64_t o0 = ((uint64_t)v[4 * mm + 1] << 32) | v[4 * mm];
                uint64_t o1 = ((uint64_t)v[4 * mm + 3] << 32) | v[4 * mm + 2];
                o0 += from_torus_f64(re[m]);
                o1 += from_torus_f64(im[m]);
                v[4 * mm] = (uint32_t)o0; v[4 * mm + 1] = (uint32_t)(o0 >> 32);
                v[4 * mm + 2] = (uint32_t)o1; v[4 * mm + 3] = (uint32_t)(o1 >> 32);
                pb[j] = o0; pb[j + kM] = o1;
                re[m] = __longlong_as_double((long long)o0);
                im[m] = __longlong_as_double((long long)o1);
            }
            tmem_st16(tmem_mine + 16 * kk, v);
        }
        tmem_wait_st();
    }

    // sample extraction (coefficient 0) straight from the registers: out[0] = A[0], out[N-j] = -A[j]; body = B[0]
    if (live) {
        uint64_t *o = out + (size_t)(out_slot ? out_slot[ct] : ct) * (kN + 1);
        if (w == 0) {
#pragma unroll
            for (int m = 0; m < 16; ++m) {
                const int j = T + 64 * m;
                const uint64_t v0 = (uint64_t)__double_as_longlong(re[m]), v1 = (uint64_t)__double_as_longlong(im[m]);
                if (j == 0) o[0] = v0; else o[kN - j] = (uint64_t)0 - v0;
                o[kN - (j + kM)] = (uint64_t)0 - v1;
            }
        } else if (T == 0) {
            o[kN] = (uint64_t)__double_as_longlong(re[0]);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (W == 0) tmem_dealloc<TMEM_COLS>(sm.tmem_base);
}

// std -> Fourier key in the v4 ring layout (64 threads per polynomial; same forward transform as the kernel above)
__global__ void __launch_bounds__(64)
bsk_convert_kernel_v4(const uint64_t *__restrict__ bsk_std, cplx *__restrict__ bskf4, const cplx *__restrict__ tbl16, int n_polys) {
    __shared__ cplx tile[kTileCplx];
    const int qd = blockIdx.x, T = threadIdx.x;
    if (qd >= n_polys) return;
    const int i = qd >> 2, r = (qd >> 1) & 1, c = qd & 1;   // std layout [i][level 1][row r][col c][N]
    const uint64_t *src = bsk_std + (size_t)qd * kN;
    const double scale = 5.293955920339377e-23;              // 2^-74
    double re[16], im[16];
#pragma unroll
    for (int m = 0; m < 16; ++m) {
        const int j = T + 64 * m;
        re[m] = DMUL((double)(long long)src[j], scale);
        im[m] = DMUL((double)(long long)src[j + kM], scale);
    }
    fft16_fwd(re, im, tile, GlobalTwiddles{tbl16, T}, T, BlockSync{});
    const int sel = (r == c) ? 0 : 1;
#pragma unroll
    for (int g = 0; g < 16; ++g) {
        cplx v; v.x = re[g]; v.y = im[g];
        bskf4[bskf4_index(i, g / QPP, c, sel, g % QPP) + T] = v;
    }
}

}  // namespace tb4

namespace tbk {

cudaError_t pbs_v4_configure() {
    cudaError_t e = cudaFuncSetAttribute(tb4::pbs_classic_kernel_v4<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tb4::Smem<4>));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(tb4::pbs_classic_kernel_v4<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tb4::Smem<3>));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(tb4::pbs_classic_kernel_v4<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tb4::Smem<2>));
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(tb4::pbs_classic_kernel_v4<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tb4::Smem<1>));
}

cudaError_t launch_pbs_classic_v4(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskf4,
                                  const void *tbl16, uint64_t *out, const uint32_t *out_slot, int batch, int n, int base_log,
                                  int n_iters, int small_is_u16, int cts, cudaStream_t stream) {
    if (batch <= 0) return cudaSuccess;
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const tb::cplx *bk = reinterpret_cast<const tb::cplx *>(bskf4), *tb = reinterpret_cast<const tb::cplx *>(tbl16);
    // cts: ciphertexts per SM the caller planned for (3 or 4), 0 = pick the instance from the batch size
    if (cts == 0 && std::getenv("TFHE_B200_WIDE_CTS") && std::getenv("TFHE_B200_WIDE_CTS")[0] == '3' && batch > 2 * sms) cts = 3;
    if (cts == 0) cts = batch <= sms ? 1 : batch <= 2 * sms ? 2 : batch <= 3 * sms ? 3 : 4;
    if (cts == 1)
        tb4::pbs_classic_kernel_v4<1><<<batch, 128, sizeof(tb4::Smem<1>), stream>>>(lwe_small, lut_idx, luts, bk, tb, out, out_slot, batch, n,
                                                                                  base_log, n_iters, small_is_u16);
    else if (cts == 2)
        tb4::pbs_classic_kernel_v4<2><<<(batch + 1) / 2, 256, sizeof(tb4::Smem<2>), stream>>>(lwe_small, lut_idx, luts, bk, tb, out, out_slot,
                                                                                            batch, n, base_log, n_iters, small_is_u16);
    else if (cts == 3)
        // one wave of three ciphertexts per SM (152 registers, 7-slot ring) takes 5.5 ms against 7.25 ms for a -- then mostly empty -- wave
        // of four; TFHE_B200_WIDE_CTS=3 runs every wide batch on this instance (the A/B that showed equal throughput from 12 and 16 warps)
        tb4::pbs_classic_kernel_v4<3><<<(batch + 2) / 3, 384, sizeof(tb4::Smem<3>), stream>>>(lwe_small, lut_idx, luts, bk, tb, out, out_slot,
                                                                                            batch, n, base_log, n_iters, small_is_u16);
    else
        tb4::pbs_classic_kernel_v4<4><<<(batch + 3) / 4, 512, sizeof(tb4::Smem<4>), stream>>>(lwe_small, lut_idx, luts, bk, tb, out, out_slot,
                                                                                            batch, n, base_log, n_iters, small_is_u16);
    return cudaGetLastError();
}

cudaError_t launch_bsk_convert_v4(const uint64_t *bsk_std, void *bskf4, const void *tbl16, int n_polys, cudaStream_t stream) {
    tb4::bsk_convert_kernel_v4<<<n_polys, 64, 0, stream>>>(bsk_std, reinterpret_cast<tb::cplx *>(bskf4),
                                                          reinterpret_cast<const tb::cplx *>(tbl16), n_polys);
    return cudaGetLastError();
}

}  // namespace tbk
