// pbs_multibit_v8.cu -- multi-bit programmable bootstrap (grouping factor 3) for NARROW tree levels (at most one ciphertext per SM):
// the arithmetic of pbs_multibit_v4.cu (lwe_multi_bit_programmable_bootstrapping.rs:18-84,295-546; fft/mod.rs:408-445;
// ggsw.rs:699-754) on the thread layout of pbs_v8.cu -- four warps per polynomial, 8 FFT points per thread (pbs8_common.cuh), eight
// warps per ciphertext -- because a narrow multi-bit level is bound by the per-thread key-combine loop (7 complex products per key
// entry and frequency): halving the frequencies per thread halves that chain.
//
// With one ciphertext per CTA everything per-thread lives in registers: the accumulator (as u64 bit patterns in the FFT registers --
// the monomials are applied in the Fourier domain, nothing is gathered), the 24 FFT twiddles and the step's seven A_j; no TMEM.
// M_j[k] = zeta_k^(deg_j), zeta_k = w^(1 - 4k), k = kT + 128*x(register), x = (r >> 2) + 2*brev2(r & 3):
//     M_j = A_j * W8^(deg_j * x),  A_j = w^(deg_j * (1 - 4*kT)) from two 64-entry root tables in shared memory.
// Key stream: 512 KiB per step through a ring of eleven 16 KiB pieces ([j & 1][out poly][sel][thread 128]: two GGSWs of ONE frequency);
// the four pieces of a frequency are released together.
#include "kernels.h"
#include "sample_extract.cuh"
#include "pbs8_common.cuh"

namespace tbm8 {
using namespace tb8c;

constexpr int GF = 3, NGGSW = 1 << GF;
constexpr int PIECE_CPLX = 1024;               // [jl 2][out poly 2][sel 2][thread 128]
constexpr int PIECE_BYTES = PIECE_CPLX * 16;   // 16 KiB
constexpr int PIECES_PER_REG = NGGSW / 2;      // 4
constexpr int PIECES_PER_ITER = 8 * PIECES_PER_REG;   // 32 = 512 KiB per group
constexpr int NSLOT = 11;
constexpr int WARPS = 8;

__constant__ double c_w8[8][2];                // exp(-2*pi*i*e/8)

struct Smem {
    cplx tile[2][tb8::kTileCplx];
    cplx ring[NSLOT][PIECE_CPLX];
    cplx root_hi[64], root_lo[64];             // w^(64 x), w^y: w^e = root_hi[e >> 6] * root_lo[e & 63]
    unsigned long long full_bar[NSLOT];
    unsigned int consumed[NSLOT];
};
static_assert(sizeof(Smem) <= 227 * 1024, "shared memory budget");

// Fourier key layout: piece = (group*8 + register g)*4 + (j >> 1); inside [j & 1][out poly c][sel][thread 128]
__device__ __forceinline__ size_t bskm8_index(int grp, int j, int g, int c, int sel) {
    return (((((size_t)(grp * 8 + g) * PIECES_PER_REG + (j >> 1)) * 2 + (j & 1)) * 2 + c) * 2 + sel) * 128;
}

__global__ void __launch_bounds__(256, 1)
pbs_multibit_kernel_v8(const uint64_t *__restrict__ lwe_small, const uint32_t *__restrict__ lut_idx, const uint64_t *__restrict__ luts,
                       const cplx *__restrict__ bskm, const cplx *__restrict__ tbl8, const cplx *__restrict__ roots,   // roots[e] = exp(i*pi*e/2048)
                       uint64_t *__restrict__ out, const uint32_t *__restrict__ out_slot, const tbk::ManyLut many, int batch, int n, int base_log, int n_groups) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Smem &sm = *reinterpret_cast<Smem *>(smem_raw);
    const int W = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int w = W >> 2, T = ((W & 3) << 5) | lane;
    const int ct = blockIdx.x < batch ? blockIdx.x : batch - 1;
    cplx *tile = sm.tile[w];
    const cplx *otile = sm.tile[w ^ 1];
    const PolySync128 poly_sync{1 + w};
    const uint64_t *lwe = lwe_small + (size_t)ct * (n + 1);
    const int total_pieces = n_groups * PIECES_PER_ITER;

    if (threadIdx.x < 64) {
        sm.root_hi[threadIdx.x] = __ldg(roots + 64 * threadIdx.x);
        sm.root_lo[threadIdx.x] = __ldg(roots + threadIdx.x);
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < NSLOT; ++s) { mbar_init(&sm.full_bar[s], 1); sm.consumed[s] = 0; }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int first = total_pieces < NSLOT ? total_pieces : NSLOT;
        for (int g = 0; g < first; ++g) {
            mbar_expect_tx(&sm.full_bar[g], PIECE_BYTES);
            tma_load_1d(sm.ring[g], bskm + (size_t)g * PIECE_CPLX, PIECE_BYTES, &sm.full_bar[g]);
        }
    }
    cplx twr[24];
#pragma unroll
    for (int k = 0; k < 24; ++k) twr[k] = __ldg(tbl8 + 24 * T + k);
    const RegTw8 twd{twr};

    // acc <- LUT * X^(-b_hat) (lwe_multi_bit_programmable_bootstrapping.rs:373-391), own coefficients only
    double re[8], im[8];
    {
        const uint32_t b_hat = modulus_switch_2n(__ldg(lwe + n)) & (2 * kN - 1);
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
            re[m] = __longlong_as_double((long long)v0);
            im[m] = __longlong_as_double((long long)v1);
        }
    }
    // exponent of the thread-dependent part of zeta_k = w^(1 - 4k): kT = frequency of register 0
    const int rot_t = (1 - 4 * freq_of8(T, 0)) & (2 * kN - 1);

    int slot = 0;
    uint32_t phase = 0;
    for (int grp = 0; grp < n_groups; ++grp) {
        // monomial degrees of the 7 non-constant GGSWs (:44-62): bit (g-1-t) of j selects mask element t; modulus switch of the SUM
        cplx A[NGGSW];
        uint32_t deg3 = 0;       // deg_j mod 8 (all the register-dependent factor needs), 3 bits per j
        {
            const uint64_t a0v = __ldg(lwe + GF * grp), a1v = __ldg(lwe + GF * grp + 1), a2v = __ldg(lwe + GF * grp + 2);
#pragma unroll
            for (int j = 1; j < NGGSW; ++j) {
                const uint64_t s = ((j & 4) ? a0v : 0) + ((j & 2) ? a1v : 0) + ((j & 1) ? a2v : 0);
                const uint32_t deg = modulus_switch_2n(s) & (2 * kN - 1);
                deg3 |= (deg & 7u) << (3 * j);
                const uint32_t e = (deg * (uint32_t)rot_t) & (2 * kN - 1);       // A_j = w^(deg * (1 - 4*kT))
                const cplx hi = sm.root_hi[e >> 6], lo = sm.root_lo[e & 63];
                A[j].x = DFMA(hi.x, lo.x, -DMUL(hi.y, lo.y));
                A[j].y = DFMA(hi.x, lo.y, DMUL(hi.y, lo.x));
            }
        }

        // decomposition of the accumulator itself (ggsw.rs:515-533 on src = acc_old), folded
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            re[m] = (double)signed_digit_l1((uint64_t)__double_as_longlong(re[m]), base_log);
            im[m] = (double)signed_digit_l1((uint64_t)__double_as_longlong(im[m]), base_log);
        }

        fft8_fwd(re, im, tile, twd, T, poly_sync);
        // park my 8 spectrum values for the partner polynomial (own exchange-A reader slots: conflict free, private)
        st8(tile + xa_rbase(T), re, im, [](int p) { return xa_roff(p); });
        __syncthreads();

        {
            const cplx *fop = otile + xa_rbase(T);
            int my_slot = 0, my_piece = 0;
#pragma unroll
            for (int g = 0; g < 8; ++g) {
                cplx Ga, Gb;
                const uint32_t x = (uint32_t)((g >> 2) + 2 * brev2(g & 3));
#pragma unroll
                for (int pc = 0; pc < PIECES_PER_REG; ++pc) {
                    const int p = g * PIECES_PER_REG + pc;
                    if (!mbar_try_wait(&sm.full_bar[slot], phase)) mbar_wait(&sm.full_bar[slot], phase);
#pragma unroll
                    for (int jl = 0; jl < 2; ++jl) {
                        const int j = pc * 2 + jl;
                        const cplx *base = sm.ring[slot] + ((jl * 2 + w) * 2) * 128 + T;
                        const cplx ga = base[0], gb = base[128];
                        if (j == 0) {
                            Ga = ga; Gb = gb;
                        } else {
                            // M = A_j * W8^(deg_j * x): monomial spectrum at this thread's frequency (fft/mod.rs:413-444)
                            const uint32_t e = (((deg3 >> (3 * j)) & 7u) * x) & 7u;
                            const double br = c_w8[e][0], bi = c_w8[e][1];
                            const double mr = DFMA(A[j].x, br, -DMUL(A[j].y, bi));
                            const double mi = DFMA(A[j].x, bi, DMUL(A[j].y, br));
                            Ga.x = DFMA(ga.x, mr, DFMA(-ga.y, mi, Ga.x));
                            Ga.y = DFMA(ga.x, mi, DFMA(ga.y, mr, Ga.y));
                            Gb.x = DFMA(gb.x, mr, DFMA(-gb.y, mi, Gb.x));
                            Gb.y = DFMA(gb.x, mi, DFMA(gb.y, mr, Gb.y));
                        }
                    }
                    if (lane == p) { my_slot = slot; my_piece = grp * PIECES_PER_ITER + p; }
                    if (++slot == NSLOT) { slot = 0; phase ^= 1u; }
                }
                // release the register's four slots (lane = piece index within the step); nothing is synchronised in between
                __syncwarp();
                if (lane >= g * PIECES_PER_REG && lane < (g + 1) * PIECES_PER_REG && atomicAdd(&sm.consumed[my_slot], 1u) == WARPS - 1) {
                    sm.consumed[my_slot] = 0;
                    const int g2 = my_piece + NSLOT;
                    if (g2 < total_pieces) {
                        __threadfence_block();
                        fence_proxy_async();
                        mbar_expect_tx(&sm.full_bar[my_slot], PIECE_BYTES);
                        tma_load_1d(sm.ring[my_slot], bskm + (size_t)g2 * PIECE_CPLX, PIECE_BYTES, &sm.full_bar[my_slot]);
                    }
                }
                // out_fft[w] = F_w * Gc[w][w] + F_{1-w} * Gc[1-w][w]
                const cplx F = fop[xa_roff(g)];
                const double fr = re[g], fi = im[g];
                double orr = DMUL(fr, Ga.x);
                orr = DFMA(-fi, Ga.y, orr);
                orr = DFMA(F.x, Gb.x, orr);
                orr = DFMA(-F.y, Gb.y, orr);
                double oi = DMUL(fr, Ga.y);
                oi = DFMA(fi, Ga.x, oi);
                oi = DFMA(F.x, Gb.y, oi);
                oi = DFMA(F.y, Gb.x, oi);
                re[g] = orr; im[g] = oi;
            }
        }
        __syncthreads();   // the partner polynomial has read my spectrum: the tile is mine again

        fft8_inv(re, im, tile, twd, T, poly_sync);

        // dst = 0; dst += G (x) src  (:503): the accumulator is REPLACED by the rounded product
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            re[m] = __longlong_as_double((long long)from_torus_f64(re[m]));
            im[m] = __longlong_as_double((long long)from_torus_f64(im[m]));
        }
    }

    if (blockIdx.x < batch && many.fn) {
        const int nf = tbx::many_fn_count(many, lut_idx, ct);
        tbx::extract_many_regs<8, 128, kN, 1>(out, out_slot[ct], nf, tbx::many_step(many, nf, kN), w, T, re, im);
    } else if (blockIdx.x < batch) {
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
}


// ---- the narrowest levels (at most SM count / 2 ciphertexts): one ciphertext on a cluster of TWO SMs, warp-specialised -----------------
// ncu on the one-SM kernel above and on a first two-SM version: a narrow multi-bit step is one long dependency chain per warp (2.7 k
// instructions at 5 cycles each: mbarrier probe -> key loads -> 7-term combination, 32 times, between two FFTs), not a bandwidth problem.
// But the combination G = G_0 + sum_j G_j * M_j depends only on the step's monomial degrees (mask elements of the input), not on the
// accumulator, so it need not sit on the accumulator's critical path:
//   * CTA rank w of the cluster owns polynomial w (pbs_classic_kernel_v8x2 in pbs_v8.cu has the reasoning and the same spectrum swap
//     through distributed shared memory) and streams only the half of the key that feeds output polynomial w;
//   * warps 4-7 ("combine warps") run ONE STEP AHEAD: they pull the key through the ring and leave the combined GGSW values of their
//     frequencies (Ga, Gb per register and thread, double buffered) in the Tensor Memory lane they share with the FFT thread of the same
//     index (tcgen05.st / tcgen05.ld: lane-private hand-over off the shared-memory pipe; the 64 KiB it would take in shared memory go to
//     the key ring, whose depth -- bytes in flight against a 2 us refill turn-around -- is what bounds a step);
//   * warps 0-3 ("FFT warps") do what a classic blind-rotation step does -- decompose, forward FFT, swap spectra, 2 x 2 multiply-accumulate
//     against the combined values, inverse FFT, round.
// Hand-offs are mbarriers (combined values full / empty inside the CTA; "spectrum landed" = the 16 KiB of st.async stores reported to an
// mbarrier in the receiving CTA).  The floating-point operations and their order are those of the one-SM kernel: identical words.
constexpr int NSLOTX = 5;
constexpr int HALF_REG_CPLX = 2048;            // one ring slot: [register of the pair 2][jj 4][sel 2][thread 128] = 32 KiB behind ONE barrier
struct SmemX2 {
    cplx tile[tb8::kTileCplx];
    cplx recv[2][8 * 128];
    cplx ring[NSLOTX][HALF_REG_CPLX];
    cplx root_hi[64], root_lo[64];
    unsigned long long full_bar[NSLOTX], empty_bar[NSLOTX], comb_full[2], comb_empty[2], spec_full[2];
    unsigned int consumed[NSLOTX];
    uint32_t tmem_base;
};
static_assert(sizeof(SmemX2) <= 227 * 1024, "shared memory budget");

constexpr int COMB_COLS = 128;     // Tensor Memory: [step parity 2][register g 8][Ga.x Ga.y Gb.x Gb.y as 8 words] per lane (= FFT thread T)

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(288, 1)
pbs_multibit_kernel_v8x2(const uint64_t *__restrict__ lwe_small, const uint32_t *__restrict__ lut_idx, const uint64_t *__restrict__ luts,
                         const cplx *__restrict__ bskm, const cplx *__restrict__ tbl8, const cplx *__restrict__ roots,
                         uint64_t *__restrict__ out, const uint32_t *__restrict__ out_slot, const tbk::ManyLut many, int batch, int n, int base_log, int n_groups) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    SmemX2 &sm = *reinterpret_cast<SmemX2 *>(smem_raw);
    const int T = threadIdx.x & 127, lane = threadIdx.x & 31;
    const bool combiner = threadIdx.x >= 128 && threadIdx.x < 256, producer = threadIdx.x >= 256;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    const int w = (int)rank;
    const int ct = blockIdx.x >> 1;
    const uint64_t *lwe = lwe_small + (size_t)ct * (n + 1);
    const int total_uses = n_groups * 8;      // ring slot uses: 4 register pairs x 2 halves per step

    if (threadIdx.x < 64) {
        sm.root_hi[threadIdx.x] = __ldg(roots + 64 * threadIdx.x);
        sm.root_lo[threadIdx.x] = __ldg(roots + threadIdx.x);
    }
    if (threadIdx.x == 0) {
        for (int s = 0; s < NSLOTX; ++s) { mbar_init(&sm.full_bar[s], 1); mbar_init(&sm.empty_bar[s], 4); sm.consumed[s] = 0; }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&sm.comb_full[s], 128); mbar_init(&sm.comb_empty[s], 128);
            mbar_init(&sm.spec_full[s], 1); mbar_expect_tx(&sm.spec_full[s], 8 * 128 * 16);     // armed for steps 0 and 1
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async();
    }
    if (threadIdx.x < 32) tb16k::tmem_alloc<COMB_COLS>(&sm.tmem_base);
    tb16k::tc_fence_before();
    __syncthreads();
    tb16k::tc_fence_after();
    // combine thread and FFT thread of the same T sit in the same TMEM lane (warp id % 4 = T / 32, same lane): the combined values are
    // handed over there, lane-private, off the shared-memory pipe and out of the shared-memory budget (which goes to a deeper key ring)
    const uint32_t comb_t = sm.tmem_base + ((uint32_t)((T >> 5) * 32) << 16);
    // both CTAs resident, barriers initialised, before anybody signals or stores into the partner's shared memory
    asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");

    if (producer) {
        // ================= producer warp: one lane keeps the key ring full (the refill is ~100 single-lane instructions per slot: on a
        // combine warp it made that warp the slowest, and the ring moves at the pace of the slowest reader) ==================================
        if (lane == 0) {
        // ring slot = half the key of a PAIR of FFT registers: use u = (grp * 4 + pair) * 2 + h holds, for registers g = 2 pair + cw (cw = 0, 1)
            // and GGSWs j = 4 h + jj, the [sel 2][thread 128] blocks of output polynomial w: [cw][jj][sel][thread] = 32 KiB behind one barrier.
            auto fill = [&](int slot, int u) {
                mbar_expect_tx(&sm.full_bar[slot], HALF_REG_CPLX * 16);
                const int h = u & 1, gbase = (u >> 1) * 2;           // gbase = grp * 8 + 2 * pair
#pragma unroll
                for (int q = 0; q < 8; ++q) {                        // q = cw * 4 + jj
                    const int j = 4 * h + (q & 3);
                    tma_load_1d(sm.ring[slot] + q * 256, bskm + (size_t)((gbase + (q >> 2)) * PIECES_PER_REG + (j >> 1)) * PIECE_CPLX + (((j & 1) * 2 + w) * 2) * 128,
                                256 * 16, &sm.full_bar[slot]);
                }
            };
            for (int u = 0; u < total_uses; ++u) {
                const int slot = u % NSLOTX;
                if (u >= NSLOTX) {
                    mbar_wait(&sm.empty_bar[slot], (uint32_t)(u / NSLOTX - 1) & 1u);
                    fence_proxy_async();
                }
                fill(slot, u);
            }
        }
    } else if (combiner) {
        // ================= combine warps: G = G_0 + sum_j G_j * M_j for the frequencies of FFT thread T, one step ahead ==================
        const int rot_t = (1 - 4 * freq_of8(T, 0)) & (2 * kN - 1);
        int slot = 0;
        uint32_t phase = 0;
        for (int grp = 0; grp < n_groups; ++grp) {
            cplx A[NGGSW];
            uint32_t deg3 = 0;
            {
                const uint64_t a0v = __ldg(lwe + GF * grp), a1v = __ldg(lwe + GF * grp + 1), a2v = __ldg(lwe + GF * grp + 2);
#pragma unroll
                for (int j = 1; j < NGGSW; ++j) {
                    const uint64_t s = ((j & 4) ? a0v : 0) + ((j & 2) ? a1v : 0) + ((j & 1) ? a2v : 0);
                    const uint32_t deg = modulus_switch_2n(s) & (2 * kN - 1);
                    deg3 |= (deg & 7u) << (3 * j);
                    const uint32_t e = (deg * (uint32_t)rot_t) & (2 * kN - 1);
                    const cplx hi = sm.root_hi[e >> 6], lo = sm.root_lo[e & 63];
                    A[j].x = DFMA(hi.x, lo.x, -DMUL(hi.y, lo.y));
                    A[j].y = DFMA(hi.x, lo.y, DMUL(hi.y, lo.x));
                }
            }
            const int b = grp & 1;
#pragma unroll
            for (int pair = 0; pair < 4; ++pair) {      // the two registers of a pair side by side: two independent accumulation chains
                cplx Ga[2], Gb[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (!mbar_try_wait(&sm.full_bar[slot], phase)) mbar_wait(&sm.full_bar[slot], phase);
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        const int j = 4 * h + jj;
#pragma unroll
                        for (int c2 = 0; c2 < 2; ++c2) {
                            const int g = 2 * pair + c2;
                            const uint32_t x = (uint32_t)((g >> 2) + 2 * brev2(g & 3));
                            const cplx *base = sm.ring[slot] + (c2 * 4 + jj) * 256 + T;
                            const cplx ga = base[0], gb = base[128];
                            if (j == 0) {
                                Ga[c2] = ga; Gb[c2] = gb;
                            } else {
                                const uint32_t e = (((deg3 >> (3 * j)) & 7u) * x) & 7u;
                                const double br = c_w8[e][0], bi = c_w8[e][1];
                                const double mr = DFMA(A[j].x, br, -DMUL(A[j].y, bi));
                                const double mi = DFMA(A[j].x, bi, DMUL(A[j].y, br));
                                Ga[c2].x = DFMA(ga.x, mr, DFMA(-ga.y, mi, Ga[c2].x));
                                Ga[c2].y = DFMA(ga.x, mi, DFMA(ga.y, mr, Ga[c2].y));
                                Gb[c2].x = DFMA(gb.x, mr, DFMA(-gb.y, mi, Gb[c2].x));
                                Gb[c2].y = DFMA(gb.x, mi, DFMA(gb.y, mr, Gb[c2].y));
                            }
                        }
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&sm.empty_bar[slot]);     // four warps out = the producer warp may refill the slot
                    if (++slot == NSLOTX) { slot = 0; phase ^= 1u; }
                }
                if (pair == 0 && grp >= 2) {      // the FFT warps are done with step grp - 2's values
                    mbar_wait(&sm.comb_empty[b], (uint32_t)((grp >> 1) - 1) & 1u);
                    tb16k::tc_fence_after();
                }
                {
                    uint32_t v[16];
#pragma unroll
                    for (int c2 = 0; c2 < 2; ++c2) {
                        tb16k::pack_cplx(Ga[c2].x, Ga[c2].y, v, 2 * c2);
                        tb16k::pack_cplx(Gb[c2].x, Gb[c2].y, v, 2 * c2 + 1);
                    }
                    tmem_st16(comb_t + (uint32_t)(b * 64 + pair * 16), v);
                }
            }
            tmem_wait_st();
            tb16k::tc_fence_before();
            mbar_arrive(&sm.comb_full[b]);
        }
    } else {
        // ================= FFT warps: the accumulator's critical path ===================================================================
        cplx *tile = sm.tile;
        const PolySync128 poly_sync{1};
        uint32_t peer_recv, peer_bar;
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(peer_recv) : "r"(smem_u32(&sm.recv[0][T])), "r"((uint32_t)(w ^ 1)));
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(peer_bar) : "r"(smem_u32(&sm.spec_full[0])), "r"((uint32_t)(w ^ 1)));
        cplx twr[24];
#pragma unroll
        for (int k = 0; k < 24; ++k) twr[k] = __ldg(tbl8 + 24 * T + k);
        const RegTw8 twd{twr};
        double re[8], im[8];
        {
            const uint32_t b_hat = modulus_switch_2n(__ldg(lwe + n)) & (2 * kN - 1);
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
                re[m] = __longlong_as_double((long long)v0);
                im[m] = __longlong_as_double((long long)v1);
            }
        }
        for (int grp = 0; grp < n_groups; ++grp) {
            const int b = grp & 1;
            const uint32_t par = (uint32_t)(grp >> 1) & 1u;
#pragma unroll
            for (int m = 0; m < 8; ++m) {
                re[m] = (double)signed_digit_l1((uint64_t)__double_as_longlong(re[m]), base_log);
                im[m] = (double)signed_digit_l1((uint64_t)__double_as_longlong(im[m]), base_log);
            }
            fft8_fwd(re, im, tile, twd, T, poly_sync);
            {   // my spectrum -> the partner's receive buffer b: the partner read it last in step grp - 2, and it finished that step's
                // multiply-accumulate before it sent me the spectrum of step grp - 1, which I have consumed
                const uint32_t dst = peer_recv + (uint32_t)(b * 8 * 128 * 16);
#pragma unroll
                for (int c = 0; c < 8; ++c) st_async_cluster(dst + (uint32_t)(c * 128 * 16), re[c], im[c], peer_bar + (uint32_t)(b * 8));
            }
            if (!mbar_try_wait(&sm.comb_full[b], par)) mbar_wait(&sm.comb_full[b], par);
            tb16k::tc_fence_after();
            const uint32_t cg = comb_t + (uint32_t)(b * 64);
#pragma unroll
            for (int gp = 0; gp < 4; ++gp) {      // the half of the product that needs only my own spectrum, while the partner's is in flight
                uint32_t v[16];
                tmem_ld16(cg + 16 * gp, v);
                tmem_wait_ld();
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int g = 2 * gp + q;
                    const cplx Ga = cplx_from_words(v, 2 * q);
                    const double fr = re[g], fi = im[g];
                    re[g] = DFMA(-fi, Ga.y, DMUL(fr, Ga.x));
                    im[g] = DFMA(fi, Ga.x, DMUL(fr, Ga.y));
                }
            }
            if (!mbar_try_wait(&sm.spec_full[b], par)) mbar_wait(&sm.spec_full[b], par);
            if (T == 0) mbar_expect_tx(&sm.spec_full[b], 8 * 128 * 16);     // re-armed for step grp + 2 (the partner sends that only after my step grp + 1)
            const cplx *fop = sm.recv[b] + T;
#pragma unroll
            for (int gp = 0; gp < 4; ++gp) {
                uint32_t v[16];
                tmem_ld16(cg + 16 * gp, v);
                tmem_wait_ld();
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int g = 2 * gp + q;
                    const cplx Gb = cplx_from_words(v, 2 * q + 1), F = fop[g * 128];
                    double orr = DFMA(F.x, Gb.x, re[g]);
                    orr = DFMA(-F.y, Gb.y, orr);
                    double oi = DFMA(F.x, Gb.y, im[g]);
                    oi = DFMA(F.y, Gb.x, oi);
                    re[g] = orr; im[g] = oi;
                }
            }
            tb16k::tc_fence_before();
            mbar_arrive(&sm.comb_empty[b]);
            fft8_inv(re, im, tile, twd, T, poly_sync);
#pragma unroll
            for (int m = 0; m < 8; ++m) {
                re[m] = __longlong_as_double((long long)from_torus_f64(re[m]));
                im[m] = __longlong_as_double((long long)from_torus_f64(im[m]));
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
    }
    // nobody leaves while the partner could still address its shared memory
    tb16k::tc_fence_before();
    asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
    if (threadIdx.x < 32) tb16k::tmem_dealloc<COMB_COLS>(sm.tmem_base);
}

// std multi-bit key [group][j 8][level 1][row r][col c][N] (entities/lwe_multi_bit_bootstrap_key.rs:11-62) -> ring layout
__global__ void __launch_bounds__(128)
bsk_convert_multibit_kernel_v8(const uint64_t *__restrict__ bsk_std, cplx *__restrict__ bskm, const cplx *__restrict__ tbl8, int n_polys) {
    __shared__ cplx tile[tb8::kTileCplx];
    const int qd = blockIdx.x, T = threadIdx.x;
    if (qd >= n_polys) return;
    const int c = qd & 1, r = (qd >> 1) & 1, j = (qd >> 2) & 7, grp = qd >> 5;
    const uint64_t *src = bsk_std + (size_t)qd * kN;
    const double scale = 5.293955920339377e-23;   // 2^-74
    double re[8], im[8];
#pragma unroll
    for (int m = 0; m < 8; ++m) {
        const int jj = T + 128 * m;
        re[m] = DMUL((double)(long long)src[jj], scale);
        im[m] = DMUL((double)(long long)src[jj + kM], scale);
    }
    fft8_fwd(re, im, tile, GlobalTw8{tbl8 + 24 * T}, T, BlockSync{});
    const int sel = (r == c) ? 0 : 1;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
        cplx v; v.x = re[g]; v.y = im[g];
        bskm[bskm8_index(grp, j, g, c, sel) + T] = v;
    }
}

}  // namespace tbm8

namespace tbk {

cudaError_t pbs_multibit_v8_configure() {
    double h[8][2];
    const long double pi = 3.14159265358979323846264338327950288L;
    for (int e = 0; e < 8; ++e) {
        h[e][0] = (double)cosl(-2.0L * pi * e / 8.0L);
        h[e][1] = (double)sinl(-2.0L * pi * e / 8.0L);
    }
    cudaError_t err = cudaMemcpyToSymbol(tbm8::c_w8, h, sizeof(h));
    if (err != cudaSuccess) return err;
    err = cudaFuncSetAttribute(tbm8::pbs_multibit_kernel_v8x2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tbm8::SmemX2));
    if (err != cudaSuccess) return err;
    return cudaFuncSetAttribute(tbm8::pbs_multibit_kernel_v8, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tbm8::Smem));
}

// one ciphertext per CTA: for batch <= SM count (the caller dispatches wider levels to launch_pbs_multibit_v4)
cudaError_t launch_pbs_multibit_v8(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskm8,
                                   const void *tbl8, const void *roots, uint64_t *out, const uint32_t *out_slot, tbk::ManyLut many, int batch, int n,
                                   int base_log, int n_groups, int cluster_max, cudaStream_t stream) {
    if (batch <= 0) return cudaSuccess;
    if (batch <= cluster_max) {
        tbm8::pbs_multibit_kernel_v8x2<<<2 * batch, 288, sizeof(tbm8::SmemX2), stream>>>(
            lwe_small, lut_idx, luts, reinterpret_cast<const tb::cplx *>(bskm8), reinterpret_cast<const tb::cplx *>(tbl8),
            reinterpret_cast<const tb::cplx *>(roots), out, out_slot, many, batch, n, base_log, n_groups);
        return cudaGetLastError();
    }
    tbm8::pbs_multibit_kernel_v8<<<batch, 256, sizeof(tbm8::Smem), stream>>>(
        lwe_small, lut_idx, luts, reinterpret_cast<const tb::cplx *>(bskm8), reinterpret_cast<const tb::cplx *>(tbl8),
        reinterpret_cast<const tb::cplx *>(roots), out, out_slot, many, batch, n, base_log, n_groups);
    return cudaGetLastError();
}

cudaError_t launch_bsk_convert_multibit_v8(const uint64_t *bsk_std, void *bskm8, const void *tbl8, int n_polys, cudaStream_t stream) {
    tbm8::bsk_convert_multibit_kernel_v8<<<n_polys, 128, 0, stream>>>(bsk_std, reinterpret_cast<tb::cplx *>(bskm8),
                                                                    reinterpret_cast<const tb::cplx *>(tbl8), n_polys);
    return cudaGetLastError();
}

}  // namespace tbk
