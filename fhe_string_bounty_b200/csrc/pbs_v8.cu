// pbs_v8.cu -- blind rotation for NARROW tree levels (at most two ciphertexts per SM): the data path of pbs_v4.cu (TMA-fed key
// ring, accumulator master copy and FFT twiddles in Tensor Memory) with FOUR warps per polynomial and 8 FFT points per thread
// (fft8_core.cuh), i.e. eight warps per ciphertext.
//
// Why: a level of <= 148 blocks puts one ciphertext on an SM.  With pbs_v4's four warps per ciphertext that is one warp per
// scheduler: ncu (scripts/narrow_level_case.py) shows issue slots 26 % busy and the warp stalled on its own instruction fetch
// (no_instruction 0.55 per instruction), fixed-latency waits (0.68) and shared-memory round trips (0.60) -- nothing to overlap
// them with.  Eight warps do half the instructions each and give every scheduler two warps.  The price (a third exchange per
// FFT, 50 % more shared-memory traffic) does not matter when the SM is otherwise idle; wide levels keep using pbs_v4.cu.
//
// Measured on a 148-block level: pbs_v4's narrow instance 4.13 ms; this kernel with all three exchanges through shared memory 4.02 ms
// (it moves 7.1 k shared-memory wavefronts per iteration against 3.6 k and becomes LSU bound, the pair exchange being 2-way bank
// conflicted); with the pair exchange done by register shuffles (exchange_c_* below) 3.52 ms.  TFHE_B200_NARROW_KERNEL=0 disables it.
//
// Same arithmetic definition as the other generations (bootstrap.rs:242-364, ggsw.rs:477-598, fft/mod.rs:197-326).
// Shared memory: 17 KiB tile per polynomial + the key ring, double buffered by whole iterations (2 x 64 KiB).
// Named barriers: 1..4 one per polynomial (128 threads), 5..6 one per ciphertext (256 threads).
#include "kernels.h"
#include "sample_extract.cuh"
#include "pbs8_common.cuh"

namespace tb8k {
using namespace tb8c;

constexpr int PIECE_CPLX = 512;        // [out poly 2][sel 2][thread 128]: one frequency (register) per thread
constexpr int PIECES_PER_ITER = 8;
constexpr int ITER_CPLX = PIECES_PER_ITER * PIECE_CPLX;   // one GGSW = one blind-rotation iteration = 64 KiB
constexpr int ITER_BYTES = ITER_CPLX * 16;
constexpr int NBUF = 2;                // the key ring is double buffered by whole iterations: one barrier, one release per iteration

template <int CTS>
struct Smem {
    cplx tile[2 * CTS][tb8::kTileCplx];    // 17 KiB per polynomial
    cplx ring[NBUF][ITER_CPLX];            // 128 KiB
    unsigned long long full_bar[NBUF];
    unsigned int consumed[NBUF];
    uint32_t tmem_base;
};
static_assert(sizeof(Smem<2>) <= 227 * 1024, "shared memory budget");


// Fourier key, v8 layout: [ggsw i][register g 8][out poly c][sel: 0 = row c, 1 = row 1-c][thread 128]
__device__ __forceinline__ size_t bskf8_index(int i, int g, int c, int sel) {
    return (((size_t)(i * PIECES_PER_ITER + g) * 2 + c) * 2 + sel) * 128;
}

template <int CTS>
__global__ void __launch_bounds__(256 * CTS, 1)
pbs_classic_kernel_v8(const uint64_t *__restrict__ lwe_small, const uint32_t *__restrict__ lut_idx, const uint64_t *__restrict__ luts,
                      const cplx *__restrict__ bskf8, const cplx *__restrict__ tbl8, uint64_t *__restrict__ out,
                      const uint32_t *__restrict__ out_slot, const tbk::ManyLut many, int batch, int n, int base_log, int n_iters, int small_is_u16) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int WARPS = 8 * CTS, TMEM_COLS = 256, TW_COL = 128;   // accumulators: 32 columns per (ciphertext, polynomial); twiddles: 96
    constexpr bool REGS = CTS == 1;     // one ciphertext per CTA: twiddles and the accumulator master copy live in registers, no TMEM
    Smem<CTS> &sm = *reinterpret_cast<Smem<CTS> *>(smem_raw);
    const int W = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // warp -> (ciphertext, polynomial, quarter of the polynomial); TMEM lane quarter = warp id % 4 = quarter of the polynomial, so
    // all warps that share a TMEM lane have the same thread index T and can share the twiddle columns
    const int ctl = W >> 3, w = (W >> 2) & 1, T = ((W & 3) << 5) | lane, P = W >> 2;
    const int ct_raw = blockIdx.x * CTS + ctl;
    const bool live = ct_raw < batch;
    const int ct = live ? ct_raw : batch - 1;        // ragged tail: recompute the last ciphertext, skip the store
    cplx *tile = sm.tile[P];
    const cplx *otile = sm.tile[P ^ 1];
    uint64_t *pb = reinterpret_cast<uint64_t *>(tile);   // the polynomial (2048 words) for the rotated gather
    const PolySync128 poly_sync{1 + P};
    const int ct_bar = 5 + ctl;
    const uint64_t *lwe = lwe_small + (size_t)ct * (n + 1);
    const uint16_t *lwe16 = reinterpret_cast<const uint16_t *>(lwe_small) + (size_t)ct * (n + 1);

    if (threadIdx.x == 0) {
        for (int s = 0; s < NBUF; ++s) { mbar_init(&sm.full_bar[s], 1); sm.consumed[s] = 0; }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async();
    }
    if (!REGS && W == 0) tmem_alloc<TMEM_COLS>(&sm.tmem_base);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_lane = REGS ? 0u : sm.tmem_base + ((uint32_t)((W & 3) * 32) << 16);
    const uint32_t tmem_mine = tmem_lane + (uint32_t)(32 * P);
    const TmemTw8 twd_t{tmem_lane + (uint32_t)TW_COL};
    cplx twr[24];
    uint64_t accr[16];
    const RegTw8 twd_r{twr};
    if (REGS) {
#pragma unroll
        for (int k = 0; k < 24; ++k) twr[k] = __ldg(tbl8 + 24 * T + k);
    } else {   // this thread's 24 twiddles -> TMEM (6 x 16 columns)
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            uint32_t v[16];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const cplx t = __ldg(tbl8 + 24 * T + 4 * k + q);
                v[4 * q] = (uint32_t)__double2loint(t.x); v[4 * q + 1] = (uint32_t)__double2hiint(t.x);
                v[4 * q + 2] = (uint32_t)__double2loint(t.y); v[4 * q + 3] = (uint32_t)__double2hiint(t.y);
            }
            tmem_st16(twd_t.col + 16 * k, v);
        }
    }
    if (threadIdx.x == 0) {
        for (int g = 0; g < NBUF && g < n_iters; ++g) {
            mbar_expect_tx(&sm.full_bar[g], ITER_BYTES);
            tma_load_1d(sm.ring[g], bskf8 + (size_t)g * ITER_CPLX, ITER_BYTES, &sm.full_bar[g]);
        }
    }

    // ---- acc <- LUT * X^(-b_hat): registers (own coefficients as u64 bit patterns in re/im), TMEM, shared ------------------------
    double re[8], im[8];
    {
        const uint32_t b_hat = (small_is_u16 ? (uint32_t)__ldg(lwe16 + n) : modulus_switch_2n(__ldg(lwe + n))) & (2 * kN - 1);
        const uint32_t a0 = (2 * kN - b_hat) & (2 * kN - 1);
        const uint64_t *lut = luts + ((size_t)(lut_idx ? lut_idx[ct] : 0) * 2 + w) * kN;
        uint32_t v[2][16];
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            const int j = T + 128 * m;
            int s0, s1; bool n0, n1;
            rot_src(j, a0, s0, n0);
            rot_src(j + kM, a0, s1, n1);
            uint64_t v0 = __ldg(lut + s0), v1 = __ldg(lut + s1);
            v0 = n0 ? (uint64_t)0 - v0 : v0;
            v1 = n1 ? (uint64_t)0 - v1 : v1;
            pb[j] = v0; pb[j + kM] = v1;
            re[m] = __longlong_as_double((long long)v0);
            im[m] = __longlong_as_double((long long)v1);
            uint32_t *d = &v[m >> 2][4 * (m & 3)];
            d[0] = (uint32_t)v0; d[1] = (uint32_t)(v0 >> 32); d[2] = (uint32_t)v1; d[3] = (uint32_t)(v1 >> 32);
            accr[2 * m] = v0; accr[2 * m + 1] = v1;
        }
        if (!REGS) {
            tmem_st16(tmem_mine, v[0]);
            tmem_st16(tmem_mine + 16, v[1]);
            tmem_wait_st();
        }
    }

    for (int i = 0; i < n_iters; ++i) {
        const uint32_t a = (small_is_u16 ? (uint32_t)__ldg(lwe16 + i) : modulus_switch_2n(__ldg(lwe + i))) & (2 * kN - 1);   // a == 0 is NOT skipped
        poly_sync();    // the accumulator polynomial is complete in shared memory

        // ct1 = acc * X^a - acc, level-1 signed digit, folded (own coefficients come from the registers)
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            const int j = T + 128 * m;
            const uint64_t o0 = (uint64_t)__double_as_longlong(re[m]), o1 = (uint64_t)__double_as_longlong(im[m]);
            const uint32_t u = ((uint32_t)j - a) << (31 - kLogN);
            uint32_t wrap0, wrap1;
            const uint64_t r0 = rot_gather(pb, u, wrap0), r1 = rot_gather(pb, u + ((uint32_t)kM << (31 - kLogN)), wrap1);
            re[m] = (double)rot_sub_digit(r0, wrap0, o0, base_log);
            im[m] = (double)rot_sub_digit(r1, wrap1, o1, base_log);
        }

        if (REGS) fft8_fwd(re, im, tile, twd_r, T, poly_sync); else fft8_fwd(re, im, tile, twd_t, T, poly_sync);

        // spectrum exchange between the two polynomials of the ciphertext: park my 8 values in my own exchange-A reader slots (conflict
        // free, private to this thread, and nobody in the half-warp still reads the tile: fft8_fwd ends with a __syncwarp)
        st8(tile + xa_rbase(T), re, im, [](int p) { return xa_roff(p); });
        bar_sync(ct_bar, 256);

        // out_fft[w] = F_w * G[w][w] + F_{1-w} * G[1-w][w].  The whole GGSW of this iteration sits in ring buffer i & 1 behind ONE
        // barrier: 24 independent 16-byte loads and 64 FP64 instructions the compiler can interleave freely, then one release; the last
        // of the WARPS warps refills the buffer with the GGSW of iteration i + 2 (a single 64 KiB bulk copy).
        {
            const int buf = i & (NBUF - 1);
            const uint32_t ph = (uint32_t)(i / NBUF) & 1u;
            if (!mbar_try_wait(&sm.full_bar[buf], ph)) mbar_wait(&sm.full_bar[buf], ph);
            const cplx *fop = otile + xa_rbase(T);
            const cplx *pc = sm.ring[buf] + (w * 2) * 128 + T;
#pragma unroll
            for (int c = 0; c < PIECES_PER_ITER; ++c) {
                const cplx A = pc[c * PIECE_CPLX], B = pc[c * PIECE_CPLX + 128], F = fop[xa_roff(c)];
                const double fr = re[c], fi = im[c];
                double orr = DMUL(fr, A.x);
                orr = DFMA(-fi, A.y, orr);
                orr = DFMA(F.x, B.x, orr);
                orr = DFMA(-F.y, B.y, orr);
                double oi = DMUL(fr, A.y);
                oi = DFMA(fi, A.x, oi);
                oi = DFMA(F.x, B.y, oi);
                oi = DFMA(F.y, B.x, oi);
                re[c] = orr; im[c] = oi;
            }
            __syncwarp();     // every lane's loads from the ring have returned (their values fed the arithmetic above)
            if (lane == 0 && atomicAdd(&sm.consumed[buf], 1u) == WARPS - 1) {
                sm.consumed[buf] = 0;
                if (i + NBUF < n_iters) {
                    __threadfence_block();
                    fence_proxy_async();
                    mbar_expect_tx(&sm.full_bar[buf], ITER_BYTES);
                    tma_load_1d(sm.ring[buf], bskf8 + (size_t)(i + NBUF) * ITER_CPLX, ITER_BYTES, &sm.full_bar[buf]);
                }
            }
        }
        bar_sync(ct_bar, 256);   // the partner polynomial has read my spectrum: the tile is mine again

        if (REGS) fft8_inv(re, im, tile, twd_r, T, poly_sync); else fft8_inv(re, im, tile, twd_t, T, poly_sync);
        poly_sync();    // everyone has read the last exchange: the tile becomes the accumulator polynomial again

        // acc += from_torus(.): master copy in TMEM (registers when REGS), new values to registers (next gather's "own") and shared
        if (REGS) {
#pragma unroll
            for (int m = 0; m < 8; ++m) {
                const int j = T + 128 * m;
                const uint64_t o0 = accr[2 * m] + from_torus_f64(re[m]), o1 = accr[2 * m + 1] + from_torus_f64(im[m]);
                accr[2 * m] = o0; accr[2 * m + 1] = o1;
                pb[j] = o0; pb[j + kM] = o1;
                re[m] = __longlong_as_double((long long)o0);
                im[m] = __longlong_as_double((long long)o1);
            }
        } else {
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                uint32_t v[16];
                tmem_ld16(tmem_mine + 16 * k, v);
                tmem_wait_ld();
#pragma unroll
                for (int mm = 0; mm < 4; ++mm) {
                    const int m = 4 * k + mm, j = T + 128 * m;
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
                tmem_st16(tmem_mine + 16 * k, v);
            }
            tmem_wait_st();
        }
    }

    // sample extraction (coefficient 0) straight from the registers: out[0] = A[0], out[N-j] = -A[j]; body = B[0]
    if (live && many.fn) {
        const int nf = tbx::many_fn_count(many, lut_idx, ct);
        tbx::extract_many_regs<8, 128, kN, 1>(out, out_slot[ct], nf, tbx::many_step(many, nf, kN), w, T, re, im);
    } else if (live) {
        uint64_t *o = out + (size_t)(out_slot ? out_slot[ct] : ct) * (kN + 1);
        if (w == 0) {
#pragma unroll
            for (int m = 0; m < 8; ++m) {
                const int j = T + 128 * m;
                const uint64_t v0 = (uint64_t)__double_as_longlong(re[m]), v1 = (uint64_t)__double_as_longlong(im[m]);
                if (j == 0) o[0] = v0; else o[kN - j] = (uint64_t)0 - v0;
                o[kN - (j + kM)] = (uint64_t)0 - v1;
            }
        } else if (T == 0) {
            o[kN] = (uint64_t)__double_as_longlong(re[0]);
        }
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (!REGS && W == 0) tmem_dealloc<TMEM_COLS>(sm.tmem_base);
}


// ---- the narrowest levels (at most SM count / 2 ciphertexts): ONE ciphertext on a CLUSTER of two SMs -------------------------------
// ncu on the one-ciphertext instance above (profiles/r01_pbs_v8_narrow_level_summary.txt): its eight warps run in lockstep between
// barriers, so an iteration costs the SUM of its shared-memory phases (4.2 k wavefronts on the SM-wide pipe) and its FP64 phases (2 warps
// per scheduler), 7.4 k cycles, with nothing to overlap.  Both halve when each polynomial gets an SM of its own: CTA rank w of the cluster
// owns polynomial w (accumulator, gather, forward FFT, the output polynomial w of the external product, inverse FFT), streams only the
// half of the Fourier key that feeds output w (8 x 4 KiB pieces per iteration into a four-deep ring), and the two CTAs swap spectra once
// per iteration: each thread stores its 8 values straight into the partner's shared memory (st.shared::cluster, double buffered) and
// every store reports its bytes to an mbarrier in the partner's shared memory (st.async ... mbarrier::complete_tx): 16 KiB received = the
// spectrum has landed.  No fence, no cluster barrier inside the loop (a cluster barrier per iteration, or 128 release.cluster arrivals,
// put a MEMBAR.ALL.GPU + ERRBAR on every thread's path: ncu, profiles/r02_pbs_v8x2_*).
constexpr int NBUFX = 4;
constexpr int SPEC_BYTES = 8 * 128 * 16;     // one polynomial's spectrum
constexpr int HALF_ITER_CPLX = PIECES_PER_ITER * 256;      // [register g 8][sel 2][thread 128] = 32 KiB
struct SmemX2 {
    cplx tile[tb8::kTileCplx];
    cplx recv[2][PIECES_PER_ITER * 128];
    cplx ring[NBUFX][HALF_ITER_CPLX];
    unsigned long long full_bar[NBUFX], empty_bar[NBUFX], spec_full[2];
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(160, 1)
pbs_classic_kernel_v8x2(const uint64_t *__restrict__ lwe_small, const uint32_t *__restrict__ lut_idx, const uint64_t *__restrict__ luts,
                        const cplx *__restrict__ bskf8, const cplx *__restrict__ tbl8, uint64_t *__restrict__ out,
                        const uint32_t *__restrict__ out_slot, const tbk::ManyLut many, int batch, int n, int base_log, int n_iters, int small_is_u16) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    SmemX2 &sm = *reinterpret_cast<SmemX2 *>(smem_raw);
    const int T = threadIdx.x;
    const int w = (int)cluster_ctarank();                 // polynomial of this CTA: 0 = mask, 1 = body
    const int ct = blockIdx.x >> 1;                       // grid = 2 * batch: every cluster has a live ciphertext
    cplx *tile = sm.tile;
    uint64_t *pb = reinterpret_cast<uint64_t *>(tile);
    const PolySync128 poly_sync{1};
    const uint64_t *lwe = lwe_small + (size_t)ct * (n + 1);
    const uint16_t *lwe16 = reinterpret_cast<const uint16_t *>(lwe_small) + (size_t)ct * (n + 1);
    const uint32_t peer_recv = map_to_cta(smem_u32(&sm.recv[0][T]), (uint32_t)(w ^ 1));
    const uint32_t peer_bar = map_to_cta(smem_u32(&sm.spec_full[0]), (uint32_t)(w ^ 1));

    auto fill = [&](int it) {      // this CTA's half of GGSW `it`: for every register g the [sel 2][thread 128] block of output polynomial w
        const int buf = it & (NBUFX - 1);
        mbar_expect_tx(&sm.full_bar[buf], HALF_ITER_CPLX * 16);
#pragma unroll
        for (int g = 0; g < PIECES_PER_ITER; ++g)
            tma_load_1d(sm.ring[buf] + g * 256, bskf8 + bskf8_index(it, g, w, 0), 256 * 16, &sm.full_bar[buf]);
    };
    if (T == 0) {
        for (int s = 0; s < NBUFX; ++s) { mbar_init(&sm.full_bar[s], 1); mbar_init(&sm.empty_bar[s], 4); }
        for (int s = 0; s < 2; ++s) { mbar_init(&sm.spec_full[s], 1); mbar_expect_tx(&sm.spec_full[s], SPEC_BYTES); }   // armed for iterations 0 and 1
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async();
    }
    cluster_sync_all();     // both CTAs are resident and their barriers initialised before anyone stores into the partner's shared memory

    if (threadIdx.x >= 128) {
        // producer warp: one lane keeps the key ring full (eight bulk copies per iteration are ~100 single-lane instructions; on an FFT
        // warp they sat on the iteration's critical path)
        if (threadIdx.x == 128) {
            for (int it = 0; it < n_iters; ++it) {
                if (it >= NBUFX) {
                    mbar_wait(&sm.empty_bar[it & (NBUFX - 1)], (uint32_t)(it / NBUFX - 1) & 1u);
                    fence_proxy_async();
                }
                fill(it);
            }
        }
        cluster_sync_all();
        return;
    }

    cplx twr[24];
    uint64_t accr[16];
    const RegTw8 twd_r{twr};
#pragma unroll
    for (int k = 0; k < 24; ++k) twr[k] = __ldg(tbl8 + 24 * T + k);

    double re[8], im[8];
    {
        const uint32_t b_hat = (small_is_u16 ? (uint32_t)__ldg(lwe16 + n) : modulus_switch_2n(__ldg(lwe + n))) & (2 * kN - 1);
        const uint32_t a0 = (2 * kN - b_hat) & (2 * kN - 1);
        const uint64_t *lut = luts + ((size_t)(lut_idx ? lut_idx[ct] : 0) * 2 + w) * kN;
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            const int j = T + 128 * m;
            int s0, s1; bool n0, n1;
            rot_src(j, a0, s0, n0);
            rot_src(j + kM, a0, s1, n1);
            uint64_t v0 = __ldg(lut + s0), v1 = __ldg(lut + s1);
            v0 = n0 ? (uint64_t)0 - v0 : v0;
            v1 = n1 ? (uint64_t)0 - v1 : v1;
            pb[j] = v0; pb[j + kM] = v1;
            re[m] = __longlong_as_double((long long)v0);
            im[m] = __longlong_as_double((long long)v1);
            accr[2 * m] = v0; accr[2 * m + 1] = v1;
        }
    }
    for (int i = 0; i < n_iters; ++i) {
        const uint32_t a = (small_is_u16 ? (uint32_t)__ldg(lwe16 + i) : modulus_switch_2n(__ldg(lwe + i))) & (2 * kN - 1);
        poly_sync();    // the accumulator polynomial is complete in shared memory
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            const int j = T + 128 * m;
            const uint32_t s0 = ((uint32_t)j - a) & (2 * kN - 1);
            const uint32_t s1 = (s0 + kM) & (2 * kN - 1);
            uint64_t r0 = pb[s0 & (kN - 1)], r1 = pb[s1 & (kN - 1)];
            r0 = (s0 >= (uint32_t)kN) ? (uint64_t)0 - r0 : r0;
            r1 = (s1 >= (uint32_t)kN) ? (uint64_t)0 - r1 : r1;
            const uint64_t o0 = (uint64_t)__double_as_longlong(re[m]), o1 = (uint64_t)__double_as_longlong(im[m]);
            re[m] = (double)signed_digit_l1(r0 - o0, base_log);
            im[m] = (double)signed_digit_l1(r1 - o1, base_log);
        }
        fft8_fwd(re, im, tile, twd_r, T, poly_sync);

        // my spectrum -> the partner's receive buffer i & 1: the partner read that buffer last in iteration i - 2, i.e. before it sent
        // me the spectrum of iteration i - 1, which I have waited for
        {
            const uint32_t dst = peer_recv + (uint32_t)((i & 1) * PIECES_PER_ITER * 128 * 16);
            const uint32_t bar = peer_bar + (uint32_t)((i & 1) * 8);      // every store reports its 16 bytes there: 16 KiB = the spectrum has landed
#pragma unroll
            for (int c = 0; c < PIECES_PER_ITER; ++c) st_async_cluster(dst + (uint32_t)(c * 128 * 16), re[c], im[c], bar);
        }

        // out_fft[w] = F_w * G[w][w] + F_{1-w} * G[1-w][w]: the half that needs only my own spectrum runs while the partner's is in flight
        {
            const int buf = i & (NBUFX - 1);
            const uint32_t ph = (uint32_t)(i / NBUFX) & 1u;
            if (!mbar_try_wait(&sm.full_bar[buf], ph)) mbar_wait(&sm.full_bar[buf], ph);
            const cplx *fop = sm.recv[i & 1] + T;
            const cplx *pc = sm.ring[buf] + T;
#pragma unroll
            for (int c = 0; c < PIECES_PER_ITER; ++c) {
                const cplx A = pc[c * 256];
                const double fr = re[c], fi = im[c];
                re[c] = DFMA(-fi, A.y, DMUL(fr, A.x));
                im[c] = DFMA(fi, A.x, DMUL(fr, A.y));
            }
            if (!mbar_try_wait(&sm.spec_full[i & 1], (uint32_t)(i >> 1) & 1u)) mbar_wait(&sm.spec_full[i & 1], (uint32_t)(i >> 1) & 1u);
            // re-arm for iteration i + 2: the partner cannot send that spectrum before it has received mine of iteration i + 1, which I
            // send only after this point
            if (T == 0) mbar_expect_tx(&sm.spec_full[i & 1], SPEC_BYTES);
#pragma unroll
            for (int c = 0; c < PIECES_PER_ITER; ++c) {
                const cplx B = pc[c * 256 + 128], F = fop[c * 128];
                double orr = DFMA(F.x, B.x, re[c]);
                orr = DFMA(-F.y, B.y, orr);
                double oi = DFMA(F.x, B.y, im[c]);
                oi = DFMA(F.y, B.x, oi);
                re[c] = orr; im[c] = oi;
            }
            __syncwarp();
            if ((T & 31) == 0) mbar_arrive(&sm.empty_bar[buf]);      // four warps out = the producer may refill this ring buffer
        }
        fft8_inv(re, im, tile, twd_r, T, poly_sync);
        poly_sync();    // everyone has read the last exchange: the tile becomes the accumulator polynomial again
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            const int j = T + 128 * m;
            const uint64_t o0 = accr[2 * m] + from_torus_f64(re[m]), o1 = accr[2 * m + 1] + from_torus_f64(im[m]);
            accr[2 * m] = o0; accr[2 * m + 1] = o1;
            pb[j] = o0; pb[j + kM] = o1;
            re[m] = __longlong_as_double((long long)o0);
            im[m] = __longlong_as_double((long long)o1);
        }
    }

    if (many.fn) {
        const int nf = tbx::many_fn_count(many, lut_idx, ct);
        tbx::extract_many_regs<8, 128, kN, 1>(out, out_slot[ct], nf, tbx::many_step(many, nf, kN), w, T, re, im);
    } else {
        uint64_t *o = out + (size_t)(out_slot ? out_slot[ct] : ct) * (kN + 1);
        if (w == 0) {
#pragma unroll
            for (int m = 0; m < 8; ++m) {
                const int j = T + 128 * m;
                const uint64_t v0 = (uint64_t)__double_as_longlong(re[m]), v1 = (uint64_t)__double_as_longlong(im[m]);
                if (j == 0) o[0] = v0; else o[kN - j] = (uint64_t)0 - v0;
                o[kN - (j + kM)] = (uint64_t)0 - v1;
            }
        } else if (T == 0) {
            o[kN] = (uint64_t)__double_as_longlong(re[0]);
        }
    }
    cluster_sync_all();     // nobody leaves while the partner could still address its shared memory
}

// std -> Fourier key in the v8 ring layout (128 threads per polynomial; same forward transform as the kernel above)
__global__ void __launch_bounds__(128)
bsk_convert_kernel_v8(const uint64_t *__restrict__ bsk_std, cplx *__restrict__ bskf8, const cplx *__restrict__ tbl8, int n_polys) {
    __shared__ cplx tile[tb8::kTileCplx];
    const int qd = blockIdx.x, T = threadIdx.x;
    if (qd >= n_polys) return;
    const int i = qd >> 2, r = (qd >> 1) & 1, c = qd & 1;   // std layout [i][level 1][row r][col c][N]
    const uint64_t *src = bsk_std + (size_t)qd * kN;
    const double scale = 5.293955920339377e-23;              // 2^-74
    double re[8], im[8];
#pragma unroll
    for (int m = 0; m < 8; ++m) {
        const int j = T + 128 * m;
        re[m] = DMUL((double)(long long)src[j], scale);
        im[m] = DMUL((double)(long long)src[j + kM], scale);
    }
    fft8_fwd(re, im, tile, GlobalTw8{tbl8 + 24 * T}, T, BlockSync{});
    const int sel = (r == c) ? 0 : 1;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
        cplx v; v.x = re[g]; v.y = im[g];
        bskf8[bskf8_index(i, g, c, sel) + T] = v;
    }
}

}  // namespace tb8k

namespace tbk {

cudaError_t pbs_v8_configure() {
    cudaError_t e = cudaFuncSetAttribute(tb8k::pbs_classic_kernel_v8<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tb8k::Smem<2>));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(tb8k::pbs_classic_kernel_v8x2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tb8k::SmemX2));
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(tb8k::pbs_classic_kernel_v8<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tb8k::Smem<1>));
}

// batch <= 2 * SM count only (the caller dispatches wider levels to launch_pbs_classic_v4)
cudaError_t launch_pbs_classic_v8(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskf8,
                                  const void *tbl8, uint64_t *out, const uint32_t *out_slot, tbk::ManyLut many, int batch, int n, int base_log,
                                  int n_iters, int small_is_u16, int cluster_max, cudaStream_t stream) {
    if (batch <= 0) return cudaSuccess;
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const tb::cplx *bk = reinterpret_cast<const tb::cplx *>(bskf8), *tb = reinterpret_cast<const tb::cplx *>(tbl8);
    if (batch <= cluster_max && batch <= sms / 2)      // one ciphertext per two-SM cluster
        tb8k::pbs_classic_kernel_v8x2<<<2 * batch, 160, sizeof(tb8k::SmemX2), stream>>>(lwe_small, lut_idx, luts, bk, tb, out, out_slot, many, batch, n,
                                                                                     base_log, n_iters, small_is_u16);
    else if (batch <= sms)
        tb8k::pbs_classic_kernel_v8<1><<<batch, 256, sizeof(tb8k::Smem<1>), stream>>>(lwe_small, lut_idx, luts, bk, tb, out, out_slot, many, batch, n,
                                                                                   base_log, n_iters, small_is_u16);
    else
        tb8k::pbs_classic_kernel_v8<2><<<(batch + 1) / 2, 512, sizeof(tb8k::Smem<2>), stream>>>(lwe_small, lut_idx, luts, bk, tb, out, out_slot, many,
                                                                                             batch, n, base_log, n_iters, small_is_u16);
    return cudaGetLastError();
}

cudaError_t launch_bsk_convert_v8(const uint64_t *bsk_std, void *bskf8, const void *tbl8, int n_polys, cudaStream_t stream) {
    tb8k::bsk_convert_kernel_v8<<<n_polys, 128, 0, stream>>>(bsk_std, reinterpret_cast<tb::cplx *>(bskf8),
                                                           reinterpret_cast<const tb::cplx *>(tbl8), n_polys);
    return cudaGetLastError();
}

}  // namespace tbk
