// pbs_multibit_v4.cu -- multi-bit programmable bootstrap (grouping factor 3), second generation: the arithmetic of
// pbs_multibit.cu (lwe_multi_bit_programmable_bootstrapping.rs:18-84,295-546; fft/mod.rs:408-445; ggsw.rs:699-754) on the
// thread layout of pbs_v4.cu -- two warps per polynomial, 16 FFT points per thread, four warps per ciphertext, FFT twiddles in
// Tensor Memory -- plus 1- and 2-ciphertext instances for narrow tree levels (the first generation always packed four
// ciphertexts per SM, so a 128-block comparison level ran on 32 SMs).
//
// Per step (one group of 3 mask elements): digits of the accumulator (it lives in the FFT registers as u64 bit patterns: the
// monomials are applied in the Fourier domain, so there is no coefficient-domain rotation and nothing to gather) -> forward FFT
// -> spectrum exchange -> for each of the thread's 16 frequencies  G = G_0 + sum_{j=1..7} G_j * M_j  with
// M_j[k] = zeta_k^(deg_j), zeta_k = w^(1 - 4k), k = kT + 64*brev4(register):  M_j = A_j * W16^(deg_j * brev4(register)),
// A_j = w^(deg_j * (1 - 4*kT)) one root-table load per thread, step and j -> 2x2 MAC -> inverse FFT -> round (replace).
// The seven A_j of a step are parked in the thread's TMEM lane and re-read two at a time, because seven complex constants
// on top of 16 complex points and the running sums do not fit 128 registers.
// Key stream: 512 KiB per step through a ring of five 16 KiB pieces ([j & 1][out poly][sel][q 2][thread 64], two GGSWs of one
// 2-frequency chunk each), fed by bulk asynchronous copies; shared memory = 8 x 17 KiB tiles + 80 KiB ring.
#include "kernels.h"
#include "sample_extract.cuh"
#include "pbs16_common.cuh"
#include <cstdlib>

namespace tbm4 {
using namespace tb16k;

constexpr int GF = 3, NGGSW = 1 << GF;
constexpr int PIECE_CPLX = 1024;               // [jl 2][out poly 2][sel 2][q 2][thread 64]
constexpr int PIECE_BYTES = PIECE_CPLX * 16;   // 16 KiB
constexpr int PIECES_PER_CHUNK = NGGSW / 2;    // 4
constexpr int CHUNKS = 8;                      // 2 FFT points each
constexpr int PIECES_PER_ITER = CHUNKS * PIECES_PER_CHUNK;   // 32 = 512 KiB per group
// ring depth: whatever shared memory is left next to the tiles (a narrow-level instance is bound by the latency of the bulk
// copies times the ring depth, not by arithmetic: 5 slots give 14 us per step, 11 slots ...

__constant__ double c_w16[16][2];              // exp(-2*pi*i*e/16)

template <int CTS>
struct Smem {
    static constexpr int NSLOT = CTS == 4 ? 5 : CTS == 3 ? 7 : CTS == 2 ? 9 : 11;
    cplx tile[2 * CTS][kTileCplx];
    cplx ring[NSLOT][PIECE_CPLX];
    cplx root_hi[64], root_lo[64];         // w^(64 x), w^y: w^e = root_hi[e >> 6] * root_lo[e & 63] (no L2 round trips per step)
    unsigned long long full_bar[NSLOT];
    unsigned int consumed[NSLOT];
    uint32_t tmem_base;
};
static_assert(sizeof(Smem<4>) <= 227 * 1024 && sizeof(Smem<3>) <= 227 * 1024 && sizeof(Smem<2>) <= 227 * 1024 && sizeof(Smem<1>) <= 227 * 1024, "shared memory budget");

// Fourier key layout: piece = (group*8 + chunk)*4 + (j >> 1); inside [j & 1][out poly c][sel][q][thread]; register g = 2*chunk + q
__device__ __forceinline__ size_t bskm4_index(int grp, int j, int chunk, int c, int sel, int q) {
    return ((((((size_t)(grp * CHUNKS + chunk) * PIECES_PER_CHUNK + (j >> 1)) * 2 + (j & 1)) * 2 + c) * 2 + sel) * 2 + q) * 64;
}

template <int CTS>
__global__ void __launch_bounds__(128 * CTS, 1)
pbs_multibit_kernel_v4(const uint64_t *__restrict__ lwe_small, const uint32_t *__restrict__ lut_idx, const uint64_t *__restrict__ luts,
                       const cplx *__restrict__ bskm, const cplx *__restrict__ tbl16, const cplx *__restrict__ roots,   // roots[e] = exp(i*pi*e/2048)
                       uint64_t *__restrict__ out, const uint32_t *__restrict__ out_slot, const tbk::ManyLut many, int batch, int n, int base_log, int n_groups) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int WARPS = 4 * CTS, TMEM_COLS = 256, NSLOT = Smem<CTS>::NSLOT;   // twiddles in columns 0..79 (shared by the ciphertexts: same thread index, same values)
    Smem<CTS> &sm = *reinterpret_cast<Smem<CTS> *>(smem_raw);
    const int W = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ctl = W >> 2, w = (W >> 1) & 1, T = ((W & 1) << 5) | lane, P = W >> 1;
    const uint32_t A_COL = 80 + 32 * ctl;             // the step's A_j of THIS ciphertext: 32 columns each
    const int ct_raw = blockIdx.x * CTS + ctl;
    const bool live = ct_raw < batch;
    const int ct = live ? ct_raw : batch - 1;
    cplx *tile = sm.tile[P];
    const cplx *otile = sm.tile[P ^ 1];
    const PolySync poly_sync{1 + P};
    const int ct_bar = 9 + ctl;
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
    if (W == 0) tmem_alloc<TMEM_COLS>(&sm.tmem_base);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_lane = sm.tmem_base + ((uint32_t)((W & 3) * 32) << 16);
    const TmemTwiddles twd{tmem_lane};
    {   // this thread's twiddles -> TMEM (T1[p][T], p = 0..15, then the three pass-2 twiddles)
#pragma unroll
        for (int k = 0; k < 5; ++k) {
            uint32_t v[16];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const cplx t = k < 4 ? __ldg(tbl16 + (4 * k + q) * 64 + T) : __ldg(tbl16 + kM + 16 * (q < 3 ? q : 0) + (T & 15));
                v[4 * q] = (uint32_t)__double2loint(t.x); v[4 * q + 1] = (uint32_t)__double2hiint(t.x);
                v[4 * q + 2] = (uint32_t)__double2loint(t.y); v[4 * q + 3] = (uint32_t)__double2hiint(t.y);
            }
            tmem_st16(twd.col + 16 * k, v);
        }
        tmem_wait_st();
    }
    if (threadIdx.x == 0) {
        const int first = total_pieces < NSLOT ? total_pieces : NSLOT;
        for (int g = 0; g < first; ++g) {
            mbar_expect_tx(&sm.full_bar[g], PIECE_BYTES);
            tma_load_1d(sm.ring[g], bskm + (size_t)g * PIECE_CPLX, PIECE_BYTES, &sm.full_bar[g]);
        }
    }

    // acc <- LUT * X^(-b_hat) (lwe_multi_bit_programmable_bootstrapping.rs:373-391), own coefficients only
    double re[16], im[16];
    {
        const uint32_t b_hat = modulus_switch_2n(__ldg(lwe + n)) & (2 * kN - 1);
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
            re[m] = __longlong_as_double((long long)v0);
            im[m] = __longlong_as_double((long long)v1);
        }
    }
    // exponent of the thread-dependent part of zeta_k = w^(1 - 4k): k = kT + 64*brev4(register), kT = brev4(T >> 2) + 16*brev2(T & 3)
    const int rot_t = (1 - 4 * (brev4(T >> 2) + 16 * brev2(T & 3))) & (2 * kN - 1);

    int slot = 0;
    uint32_t phase = 0;
    for (int grp = 0; grp < n_groups; ++grp) {
        // monomial degrees of the 7 non-constant GGSWs (:44-62): bit (g-1-t) of j selects mask element t; modulus switch of the SUM.
        // A_j -> TMEM columns 80 + 4j (j = 0 slot unused); deg_j mod 16 (all the register-dependent factor needs) packed in one word.
        uint32_t deg4 = 0;
        {
            const uint64_t a0v = __ldg(lwe + GF * grp), a1v = __ldg(lwe + GF * grp + 1), a2v = __ldg(lwe + GF * grp + 2);
            uint32_t v[2][16];
#pragma unroll
            for (int j = 0; j < NGGSW; ++j) {
                cplx A; A.x = 1.0; A.y = 0.0;
                if (j > 0) {
                    const uint64_t s = ((j & 4) ? a0v : 0) + ((j & 2) ? a1v : 0) + ((j & 1) ? a2v : 0);
                    const uint32_t deg = modulus_switch_2n(s) & (2 * kN - 1);
                    deg4 |= (deg & 15u) << (4 * j);
                    const uint32_t e = (deg * (uint32_t)rot_t) & (2 * kN - 1);       // A_j = w^(deg * (1 - 4*kT))
                    const cplx hi = sm.root_hi[e >> 6], lo = sm.root_lo[e & 63];
                    A.x = DFMA(hi.x, lo.x, -DMUL(hi.y, lo.y));
                    A.y = DFMA(hi.x, lo.y, DMUL(hi.y, lo.x));
                }
                uint32_t *d = &v[j >> 2][4 * (j & 3)];
                d[0] = (uint32_t)__double2loint(A.x); d[1] = (uint32_t)__double2hiint(A.x);
                d[2] = (uint32_t)__double2loint(A.y); d[3] = (uint32_t)__double2hiint(A.y);
            }
            tmem_st16(tmem_lane + A_COL, v[0]);
            tmem_st16(tmem_lane + A_COL + 16, v[1]);
            tmem_wait_st();
        }

        // decomposition of the accumulator itself (ggsw.rs:515-533 on src = acc_old), folded
#pragma unroll
        for (int m = 0; m < 16; ++m) {
            re[m] = (double)signed_digit_l1((uint64_t)__double_as_longlong(re[m]), base_log);
            im[m] = (double)signed_digit_l1((uint64_t)__double_as_longlong(im[m]), base_log);
        }

        fft16_fwd(re, im, tile, twd, T, poly_sync);
        {   // park my 16 spectrum values in my own exchange-B reader slots for the partner polynomial
            cplx *wp = tile + xb_rbase(T);
#pragma unroll
            for (int g = 0; g < 16; ++g) { cplx v; v.x = re[g]; v.y = im[g]; wp[xb_roff(g)] = v; }
        }
        bar_sync(ct_bar, 128);

        {
            const cplx *fop = otile + xb_rbase(T);
            int my_slot = 0, my_piece = 0;
            // (measured: software-pipelining the loads of piece p+1 under piece p's arithmetic does not help -- 37.9 vs 36.3 ms for the
            // 128-char comparison -- the narrow-level instances are bound by key delivery, hence their deeper rings)
            cplx gq[2][2][2];         // [jl][sel][q]
            uint32_t av[8];           // the piece's two A_j as TMEM words
            auto load_piece = [&](int pc, int sl, uint32_t ph) {
                tmem_ld8(tmem_lane + A_COL + 8 * pc, av);
                mbar_wait(&sm.full_bar[sl], ph);
#pragma unroll
                for (int jl = 0; jl < 2; ++jl) {
                    const cplx *base = sm.ring[sl] + ((jl * 2 + w) * 2) * 2 * 64 + T;
#pragma unroll
                    for (int q = 0; q < 2; ++q) { gq[jl][0][q] = base[q * 64]; gq[jl][1][q] = base[(2 + q) * 64]; }
                }
            };
#pragma unroll
            for (int c = 0; c < CHUNKS; ++c) {
                cplx Ga[2], Gb[2];
#pragma unroll
                for (int pc = 0; pc < PIECES_PER_CHUNK; ++pc) {
                    const int p = c * PIECES_PER_CHUNK + pc;
                    load_piece(pc, slot, phase);
                    tmem_wait_ld();
                    cplx A[2];
#pragma unroll
                    for (int jl = 0; jl < 2; ++jl) {
                        A[jl].x = __hiloint2double((int)av[4 * jl + 1], (int)av[4 * jl]);
                        A[jl].y = __hiloint2double((int)av[4 * jl + 3], (int)av[4 * jl + 2]);
                    }
#pragma unroll
                    for (int jl = 0; jl < 2; ++jl) {
                        const int j = pc * 2 + jl;
#pragma unroll
                        for (int q = 0; q < 2; ++q) {
                            const cplx ga = gq[jl][0][q], gb = gq[jl][1][q];
                            if (j == 0) {
                                Ga[q] = ga; Gb[q] = gb;
                            } else {
                                // M = A_j * W16^(deg_j * brev4(g)): monomial spectrum at this thread's frequency (fft/mod.rs:413-444)
                                const int g = 2 * c + q;
                                const uint32_t e = (((deg4 >> (4 * j)) & 15u) * (uint32_t)brev4(g)) & 15u;
                                const double br = c_w16[e][0], bi = c_w16[e][1];
                                const double mr = DFMA(A[jl].x, br, -DMUL(A[jl].y, bi));
                                const double mi = DFMA(A[jl].x, bi, DMUL(A[jl].y, br));
                                Ga[q].x = DFMA(ga.x, mr, DFMA(-ga.y, mi, Ga[q].x));
                                Ga[q].y = DFMA(ga.x, mi, DFMA(ga.y, mr, Ga[q].y));
                                Gb[q].x = DFMA(gb.x, mr, DFMA(-gb.y, mi, Gb[q].x));
                                Gb[q].y = DFMA(gb.x, mi, DFMA(gb.y, mr, Gb[q].y));
                            }
                        }
                    }
                    if (lane == p) { my_slot = slot; my_piece = grp * PIECES_PER_ITER + p; }
                    if (++slot == NSLOT) { slot = 0; phase ^= 1u; }
                }
                // release the chunk's four slots (lane = piece index within the step); with only NSLOT pieces of lookahead the re-arm
                // cannot wait for the end of the step.  Nothing is synchronised inside a chunk.
                __syncwarp();
                if (lane >= c * PIECES_PER_CHUNK && lane < (c + 1) * PIECES_PER_CHUNK && atomicAdd(&sm.consumed[my_slot], 1u) == WARPS - 1) {
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
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int g = 2 * c + q;
                    const cplx F = fop[xb_roff(g)];
                    const double fr = re[g], fi = im[g];
                    double orr = DMUL(fr, Ga[q].x);
                    orr = DFMA(-fi, Ga[q].y, orr);
                    orr = DFMA(F.x, Gb[q].x, orr);
                    orr = DFMA(-F.y, Gb[q].y, orr);
                    double oi = DMUL(fr, Ga[q].y);
                    oi = DFMA(fi, Ga[q].x, oi);
                    oi = DFMA(F.x, Gb[q].y, oi);
                    oi = DFMA(F.y, Gb[q].x, oi);
                    re[g] = orr; im[g] = oi;
                }
            }
        }
        bar_sync(ct_bar, 128);   // the partner polynomial has read my spectrum: the tile is mine again

        fft16_inv(re, im, tile, twd, T, poly_sync);

        // dst = 0; dst += G (x) src  (:503): the accumulator is REPLACED by the rounded product
#pragma unroll
        for (int m = 0; m < 16; ++m) {
            re[m] = __longlong_as_double((long long)from_torus_f64(re[m]));
            im[m] = __longlong_as_double((long long)from_torus_f64(im[m]));
        }
    }

    if (live && many.fn) {
        const int nf = tbx::many_fn_count(many, lut_idx, ct);
        tbx::extract_many_regs<16, 64, kN, 1>(out, out_slot[ct], nf, tbx::many_step(many, nf, kN), w, T, re, im);
    } else if (live) {
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

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (W == 0) tmem_dealloc<TMEM_COLS>(sm.tmem_base);
}

// std multi-bit key [group][j 8][level 1][row r][col c][N] (entities/lwe_multi_bit_bootstrap_key.rs:11-62) -> ring layout
__global__ void __launch_bounds__(64)
bsk_convert_multibit_kernel_v4(const uint64_t *__restrict__ bsk_std, cplx *__restrict__ bskm, const cplx *__restrict__ tbl16, int n_polys) {
    __shared__ cplx tile[kTileCplx];
    const int qd = blockIdx.x, T = threadIdx.x;
    if (qd >= n_polys) return;
    const int c = qd & 1, r = (qd >> 1) & 1, j = (qd >> 2) & 7, grp = qd >> 5;
    const uint64_t *src = bsk_std + (size_t)qd * kN;
    const double scale = 5.293955920339377e-23;   // 2^-74
    double re[16], im[16];
#pragma unroll
    for (int m = 0; m < 16; ++m) {
        const int jj = T + 64 * m;
        re[m] = DMUL((double)(long long)src[jj], scale);
        im[m] = DMUL((double)(long long)src[jj + kM], scale);
    }
    fft16_fwd(re, im, tile, GlobalTwiddles{tbl16, T}, T, BlockSync{});
    const int sel = (r == c) ? 0 : 1;
#pragma unroll
    for (int g = 0; g < 16; ++g) {
        cplx v; v.x = re[g]; v.y = im[g];
        bskm[bskm4_index(grp, j, g >> 1, c, sel, g & 1) + T] = v;
    }
}

}  // namespace tbm4

namespace tbk {

cudaError_t pbs_multibit_v4_configure() {
    double h[16][2];
    const long double pi = 3.14159265358979323846264338327950288L;
    for (int e = 0; e < 16; ++e) {
        h[e][0] = (double)cosl(-2.0L * pi * e / 16.0L);
        h[e][1] = (double)sinl(-2.0L * pi * e / 16.0L);
    }
    cudaError_t err = cudaMemcpyToSymbol(tbm4::c_w16, h, sizeof(h));
    if (err != cudaSuccess) return err;
    err = cudaFuncSetAttribute(tbm4::pbs_multibit_kernel_v4<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tbm4::Smem<4>));
    if (err != cudaSuccess) return err;
    err = cudaFuncSetAttribute(tbm4::pbs_multibit_kernel_v4<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tbm4::Smem<3>));
    if (err != cudaSuccess) return err;
    err = cudaFuncSetAttribute(tbm4::pbs_multibit_kernel_v4<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tbm4::Smem<2>));
    if (err != cudaSuccess) return err;
    return cudaFuncSetAttribute(tbm4::pbs_multibit_kernel_v4<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tbm4::Smem<1>));
}

cudaError_t launch_pbs_multibit_v4(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskm,
                                   const void *tbl16, const void *roots, uint64_t *out, const uint32_t *out_slot, tbk::ManyLut many, int batch, int n,
                                   int base_log, int n_groups, cudaStream_t stream) {
    if (batch <= 0) return cudaSuccess;
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const tb::cplx *bk = reinterpret_cast<const tb::cplx *>(bskm), *tb = reinterpret_cast<const tb::cplx *>(tbl16),
                   *rt = reinterpret_cast<const tb::cplx *>(roots);
    // ciphertexts per CTA: 1 / 2 for narrow levels; wide levels run THREE per SM (12 warps, ring of 7 pieces): measured 92.6 ms per 8192
    // against 99.7 ms with four per SM and a ring of 5 -- the key stream (512 KiB per step) wants the shared memory more than a fourth
    // ciphertext does.  TFHE_B200_MB_CTS = 1..4 forces an instance.
    const char *fe = std::getenv("TFHE_B200_MB_CTS");
    const int force = fe ? atoi(fe) : 0;
    const int cts = force ? force : batch <= sms ? 1 : batch <= 2 * sms ? 2 : 3;
    if (cts == 1)
        tbm4::pbs_multibit_kernel_v4<1><<<batch, 128, sizeof(tbm4::Smem<1>), stream>>>(lwe_small, lut_idx, luts, bk, tb, rt, out, out_slot, many, batch,
                                                                                    n, base_log, n_groups);
    else if (cts == 2)
        tbm4::pbs_multibit_kernel_v4<2><<<(batch + 1) / 2, 256, sizeof(tbm4::Smem<2>), stream>>>(lwe_small, lut_idx, luts, bk, tb, rt, out,
                                                                                              out_slot, many, batch, n, base_log, n_groups);
    else if (cts == 3)
        tbm4::pbs_multibit_kernel_v4<3><<<(batch + 2) / 3, 384, sizeof(tbm4::Smem<3>), stream>>>(lwe_small, lut_idx, luts, bk, tb, rt, out,
                                                                                              out_slot, many, batch, n, base_log, n_groups);
    else
        tbm4::pbs_multibit_kernel_v4<4><<<(batch + 3) / 4, 512, sizeof(tbm4::Smem<4>), stream>>>(lwe_small, lut_idx, luts, bk, tb, rt, out,
                                                                                              out_slot, many, batch, n, base_log, n_groups);
    return cudaGetLastError();
}

cudaError_t launch_bsk_convert_multibit_v4(const uint64_t *bsk_std, void *bskm, const void *tbl16, int n_polys, cudaStream_t stream) {
    tbm4::bsk_convert_multibit_kernel_v4<<<n_polys, 64, 0, stream>>>(bsk_std, reinterpret_cast<tb::cplx *>(bskm),
                                                                    reinterpret_cast<const tb::cplx *>(tbl16), n_polys);
    return cudaGetLastError();
}

}  // namespace tbk
