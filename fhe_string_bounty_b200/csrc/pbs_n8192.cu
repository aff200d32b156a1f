// pbs_n8192.cu -- tuned blind rotation for N = 8192, k = 1, two PBS levels: PARAM_MESSAGE_3_CARRY_3_KS_PBS and its siblings 1_5 / 2_4 / 4_2
// (shortint/parameters/mod.rs:823-882), the third row of the reference's benchmark table (docs/getting_started/benchmarks.md:42).
//
// The generic kernel (pbs_generic.cu) runs this shape at 0.14 of the FP64 peak: the accumulator (128 KiB) and one transform buffer (64 KiB)
// fill the shared memory of an SM, so the 453 MB key comes through __ldg per ciphertext (no ring, 0.7 G spill instructions, L2 latency on
// the multiply-accumulate).  Here ONE ciphertext runs on a thread-block CLUSTER of two SMs, the layout of the narrow-level cluster kernels
// (pbs_v8.cu) at full width:
//   * CTA rank w owns polynomial w: rotated gather + two-level signed decomposition, the two forward FFTs of its own polynomial, output
//     polynomial w of the external product, the inverse FFT, the accumulator update.  Shared memory per SM = one 68 KiB tile (accumulator
//     polynomial for the gather, then FFT exchange tile) + 64 KiB landing buffer + an 80 KiB key ring.
//   * 256 threads x 16 points: FFT-4096 = radix-16, exchange A (across the CTA), radix-16, exchange B (inside a half-warp), radix-16.
//   * the key half that feeds output polynomial w ([level][own row, partner row][register][thread], contiguous per CTA) streams through
//     a TMA ring of 16 KiB pieces: 256 KiB per iteration and SM instead of 512 KiB per ciphertext through L2.
//   * per level the spectra cross the SMs once: st.async into the partner's landing buffer with mbarrier complete_tx (64 KiB), the half
//     of the multiply-accumulate that needs only the thread's own spectrum runs meanwhile; the landing buffer is single (shared memory),
//     so its release goes back as one remote mbarrier arrival per level.
//   * accumulator master copy and the 32 per-thread twiddles in Tensor Memory; the level-1 digits wait in 16 registers as packed int16.
// Same arithmetic definition as the other kernels (bootstrap.rs:242-364, ggsw.rs:477-598 levels l..1, math/decomposition.rs:25-86).
//
// FFT: point j = T + 256 m, T = u + 16 v; Z_k = sum_j z_j w^j W^(jk), w = exp(i pi / 8192), W = exp(-2 pi i / 4096), k = k1 + 16 k2 + 256 k3:
//   pass 1  radix-16 DIF over m of z w^(256 m) (pre-twist exp(i pi m / 32), as fft16_core.cuh)     -> register p1 = brev4(k1)
//   twiddle T1[p1][T] = w^T W^(T k1) = exp(i pi T (1 - 4 k1) / 8192)
//   exchange A: (T = u + 16 v, p1) -> thread T' = u + 16 p1, register v            slot 272 p1 + T
//   pass 2  radix-16 DIF over v                                                     -> register p2 = brev4(k2)
//   twiddle T2[p2][u] = W256^(u k2)
//   exchange B: (T' = u + 16 p1, p2) -> thread T'' = p2 + 16 p1, register u        slot 272 p1 + 17 p2 + u  (inside the half-warp)
//   pass 3  radix-16 DIF over u                                                     -> register p3 = brev4(k3)
#include <cstdlib>

#include "kernels.h"
#include "sample_extract.cuh"
#include "pbs16_common.cuh"
#include "fft16x_slots.cuh"

namespace tb8192 {
using namespace tb16k;
using namespace tb16x;

constexpr int LOGN = 13, N = 1 << LOGN, M = N / 2, LEVELS = 2;
constexpr int THREADS = 256;
constexpr int TILE = kTile4096;                      // 4352 complex = 68 KiB (>= N u64 words for the rotated gather)
constexpr int QPP = 4;
constexpr int PIECE_CPLX = QPP * THREADS;            // [q 4][thread 256] = 16 KiB
constexpr int PIECE_BYTES = PIECE_CPLX * 16;
constexpr int CHUNKS = 16 / QPP;
constexpr int PIECES_PER_ITER = LEVELS * 2 * CHUNKS; // [level slot][own / partner row][chunk] = 16
constexpr int NS = 5;
constexpr int SPEC_BYTES = M * 16;                   // one polynomial's spectrum: 64 KiB

struct Smem {
    cplx tile[TILE];
    cplx recv[M];
    cplx ring[NS][PIECE_CPLX];
    unsigned long long full_bar[NS], recv_full, peer_free;
    unsigned int consumed[NS];
    uint32_t tmem_base;
};
static_assert(sizeof(Smem) <= 227 * 1024, "shared memory budget");

__device__ __forceinline__ uint32_t mod_switch(uint64_t x) { return (uint32_t)(((x >> (64 - LOGN - 2)) + 1) >> 1) & (2 * N - 1); }

// the two signed digits of x (level 2 = least significant first in the carry chain): decomposer.rs:98-118, iter.rs:120-127
__device__ __forceinline__ void signed_digits2(uint64_t x, int base_log, int &d2, int &d1) {
    // base_log * LEVELS <= 31: everything the decomposition looks at sits in the top 32 bits (+ the rounding bit below), 32-bit arithmetic
    const int bits = base_log * LEVELS;
    const uint32_t hi = (uint32_t)(x >> 32);
    uint32_t state = (((hi >> (31 - bits)) + 1u) >> 1) & (bits == 31 ? 0x7FFFFFFFu : ((1u << bits) - 1u));   // closest representable, as an integer
    const uint32_t mask = (1u << base_log) - 1u;
    uint32_t digit = state & mask;
    state >>= base_log;
    uint32_t carry = (((digit - 1u) | state) & digit) >> (base_log - 1);
    state += carry;
    d2 = (int)(digit - (carry << base_log));
    digit = state & mask;
    state >>= base_log;
    carry = (((digit - 1u) | state) & digit) >> (base_log - 1);
    d1 = (int)(digit - (carry << base_log));
}

template <class Tw>
struct Fft4096 {
    // forward: on entry the tile may still be read by other threads (the first barrier covers that)
    template <class Sync>
    __device__ __forceinline__ static void fwd(double (&re)[16], double (&im)[16], cplx *tile, const Tw &twd, int T, Sync sync) {
        radix16_twisted_fwd(re, im);
        twd.template apply1<false>(re, im);
        sync();
#pragma unroll
        for (int p = 0; p < 16; ++p) { cplx v; v.x = re[p]; v.y = im[p]; tile[s4096_a_write(T, p)] = v; }
        sync();
#pragma unroll
        for (int v = 0; v < 16; ++v) { const cplx x = tile[s4096_a_read(T, v)]; re[v] = x.x; im[v] = x.y; }
        radix16_fwd(re, im);
        twd.template apply2<false>(re, im);
        __syncwarp();        // everything below stays inside the half-warp's region of the tile
#pragma unroll
        for (int p = 0; p < 16; ++p) { cplx v; v.x = re[p]; v.y = im[p]; tile[s4096_b_write(T, p)] = v; }
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 16; ++q) { const cplx x = tile[s4096_b_read(T, q)]; re[q] = x.x; im[q] = x.y; }
        radix16_fwd(re, im);
    }
    // inverse, scaled by 4096; on entry nobody may still be reading the tile, on exit it may still be read by other threads
    template <class Sync>
    __device__ __forceinline__ static void inv(double (&re)[16], double (&im)[16], cplx *tile, const Tw &twd, int T, Sync sync) {
        radix16_dit_inv(re, im);
#pragma unroll
        for (int q = 0; q < 16; ++q) { cplx v; v.x = re[q]; v.y = im[q]; tile[s4096_b_read(T, q)] = v; }
        __syncwarp();
#pragma unroll
        for (int p = 0; p < 16; ++p) { const cplx x = tile[s4096_b_write(T, p)]; re[p] = x.x; im[p] = x.y; }
        twd.template apply2<true>(re, im);
        radix16_dit_inv(re, im);
        __syncwarp();
#pragma unroll
        for (int v = 0; v < 16; ++v) { cplx x; x.x = re[v]; x.y = im[v]; tile[s4096_a_read(T, v)] = x; }
        sync();
#pragma unroll
        for (int p = 0; p < 16; ++p) { const cplx x = tile[s4096_a_write(T, p)]; re[p] = x.x; im[p] = x.y; }
        twd.template apply1<true>(re, im);
        radix16_dit_inv(re, im);
        posttwist16_inv(re, im);
    }
};

template <bool INV>
__device__ __forceinline__ void mul_tw(double &a, double &b, const cplx w) {
    const double x = a, y = b;
    if (!INV) { a = DFMA(x, w.x, -DMUL(y, w.y)); b = DFMA(y, w.x, DMUL(x, w.y)); }
    else { a = DFMA(x, w.x, DMUL(y, w.y)); b = DFMA(y, w.x, -DMUL(x, w.y)); }
}
struct TmemTw {          // T1 at col1 (64 columns, per thread), T2 at col2 (64 columns)
    uint32_t col1, col2;
    template <bool INV>
    __device__ __forceinline__ void apply(uint32_t col, double (&re)[16], double (&im)[16]) const {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            uint32_t v[16];
            tmem_ld16(col + 16 * k, v);
            tmem_wait_ld();
#pragma unroll
            for (int q = 0; q < 4; ++q) mul_tw<INV>(re[4 * k + q], im[4 * k + q], cplx_from_words(v, q));
        }
    }
    template <bool INV> __device__ __forceinline__ void apply1(double (&re)[16], double (&im)[16]) const { apply<INV>(col1, re, im); }
    template <bool INV> __device__ __forceinline__ void apply2(double (&re)[16], double (&im)[16]) const { apply<INV>(col2, re, im); }
};
struct GlobalTw {        // tbl: T1[p1 * 256 + T] (4096 entries) then T2[p2 * 16 + u] (256 entries)
    const cplx *tbl;
    int T;
    template <bool INV> __device__ __forceinline__ void apply1(double (&re)[16], double (&im)[16]) const {
#pragma unroll
        for (int p = 0; p < 16; ++p) mul_tw<INV>(re[p], im[p], __ldg(tbl + p * 256 + T));
    }
    template <bool INV> __device__ __forceinline__ void apply2(double (&re)[16], double (&im)[16]) const {
#pragma unroll
        for (int p = 0; p < 16; ++p) mul_tw<INV>(re[p], im[p], __ldg(tbl + 4096 + p * 16 + (T & 15)));
    }
};
struct CtaSync {
    __device__ __forceinline__ void operator()() const { bar_sync(1, THREADS); }
};

__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t map_peer(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_async(uint32_t addr, double x, double y, uint32_t remote_bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f64 [%0], {%1, %2}, [%3];" ::"r"(addr), "d"(x), "d"(y), "r"(remote_bar)
                 : "memory");
}
__device__ __forceinline__ void remote_arrive(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void wait_cluster(void *bar, uint32_t parity) {      // acquire at cluster scope (pairs with remote_arrive)
    const long long t0 = clock64();
    uint32_t ok = 0;
    while (!ok) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (!ok && clock64() - t0 > 4000000000LL) __trap();
    }
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// key, per output polynomial w: [w 2][ggsw i][level slot: 0 = level 2, 1 = level 1][sel: 0 = row w, 1 = row 1 - w][chunk 4][q 4][thread 256]
__device__ __forceinline__ size_t key_piece(int n_ggsw, int w, int i, int lvslot, int sel, int chunk) {
    return ((((size_t)w * n_ggsw + i) * LEVELS + lvslot) * 2 + sel) * CHUNKS + chunk;
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
pbs_n8192_kernel(const uint64_t *__restrict__ lwe_small, const uint32_t *__restrict__ lut_idx, const uint64_t *__restrict__ luts,
                 const cplx *__restrict__ bskf, const cplx *__restrict__ tbl, uint64_t *__restrict__ out,
                 const uint32_t *__restrict__ out_slot, const tbk::ManyLut many, int n, int base_log, int n_iters, int n_ggsw) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Smem &sm = *reinterpret_cast<Smem *>(smem_raw);
    const int T = threadIdx.x, W = T >> 5, lane = T & 31;
    const int w = (int)cluster_rank();
    const int ct = blockIdx.x >> 1;
    cplx *tile = sm.tile;
    uint64_t *pb = reinterpret_cast<uint64_t *>(tile);
    const CtaSync cta_sync{};
    const uint64_t *lwe = lwe_small + (size_t)ct * (n + 1);
    const cplx *key = bskf + key_piece(n_ggsw, w, 0, 0, 0, 0) * PIECE_CPLX;      // this CTA's contiguous stream of pieces
    const int total_pieces = n_iters * PIECES_PER_ITER;
    const uint32_t peer_recv = map_peer(smem_u32(&sm.recv[T]), (uint32_t)(w ^ 1));
    const uint32_t peer_full = map_peer(smem_u32(&sm.recv_full), (uint32_t)(w ^ 1));
    const uint32_t peer_peer_free = map_peer(smem_u32(&sm.peer_free), (uint32_t)(w ^ 1));

    if (T == 0) {
        for (int s = 0; s < NS; ++s) { mbar_init(&sm.full_bar[s], 1); sm.consumed[s] = 0; }
        mbar_init(&sm.recv_full, 1);
        mbar_expect_tx(&sm.recv_full, SPEC_BYTES);        // armed for the first spectrum
        mbar_init(&sm.peer_free, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async();
    }
    if (W == 0) tmem_alloc<512>(&sm.tmem_base);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    // TMEM lane quarter = warp % 4; two warps share a quarter: [accumulator 64 | T1 64] per warp, then T2 (64, shared: it depends on T & 15)
    const uint32_t quarter = sm.tmem_base + ((uint32_t)((W & 3) * 32) << 16);
    const uint32_t tmem_acc = quarter + (uint32_t)((W >> 2) * 128);
    const TmemTw twd{tmem_acc + 64, quarter + 256};
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
        uint32_t v1[16], v2[16];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const cplx a = __ldg(tbl + (4 * kk + q) * 256 + T), b = __ldg(tbl + 4096 + (4 * kk + q) * 16 + (T & 15));
            pack_cplx(a.x, a.y, v1, q);
            pack_cplx(b.x, b.y, v2, q);
        }
        tmem_st16(twd.col1 + 16 * kk, v1);
        tmem_st16(twd.col2 + 16 * kk, v2);
    }
    if (T == 0) {
        const int first = total_pieces < NS ? total_pieces : NS;
        for (int g = 0; g < first; ++g) {
            mbar_expect_tx(&sm.full_bar[g], PIECE_BYTES);
            tma_load_1d(sm.ring[g], key + (size_t)g * PIECE_CPLX, PIECE_BYTES, &sm.full_bar[g]);
        }
    }

    // ---- acc <- LUT * X^(-b_hat) ------------------------------------------------------------------------------------------------
    double re[16], im[16];
    {
        const uint32_t a0 = (2 * N - mod_switch(__ldg(lwe + n))) & (2 * N - 1);
        const uint64_t *lut = luts + ((size_t)(lut_idx ? lut_idx[ct] : 0) * 2 + w) * N;
#pragma unroll
        for (int m = 0; m < 16; ++m) {
            const int j = T + 256 * m;
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
            tmem_st16(tmem_acc + 16 * kk, v);
        }
        tmem_wait_st();
    }
    cluster_sync_all();      // both CTAs resident, barriers initialised and armed

    int slot = 0;
    uint32_t phase = 0;
    uint32_t use = 0;        // spectrum hand-overs so far (two per iteration)
    // one multiply-accumulate half: o += F * G over the four pieces of (level slot, sel); F from registers (own) or the landing buffer
    auto mac_half = [&](double (&ore)[16], double (&oim)[16], const double (&fre)[16], const double (&fim)[16], bool from_recv, int piece0) {
        int my_slot = 0;
#pragma unroll
        for (int c = 0; c < CHUNKS; ++c) {
            if (!mbar_try_wait(&sm.full_bar[slot], phase)) mbar_wait(&sm.full_bar[slot], phase);
            const cplx *pc = sm.ring[slot] + T;
#pragma unroll
            for (int q = 0; q < QPP; ++q) {
                const int g = QPP * c + q;
                const cplx G = pc[q * THREADS];
                double fr, fi;
                if (from_recv) { const cplx F = sm.recv[g * THREADS + T]; fr = F.x; fi = F.y; } else { fr = fre[g]; fi = fim[g]; }
                ore[g] = DFMA(fr, G.x, DFMA(-fi, G.y, ore[g]));
                oim[g] = DFMA(fr, G.y, DFMA(fi, G.x, oim[g]));
            }
            if (lane == c) my_slot = slot;
            if (++slot == NS) { slot = 0; phase ^= 1u; }
        }
        __syncwarp();
        if (lane < CHUNKS && atomicAdd(&sm.consumed[my_slot], 1u) == THREADS / 32 - 1) {
            sm.consumed[my_slot] = 0;
            const int k2 = piece0 + lane + NS;
            if (k2 < total_pieces) {
                __threadfence_block();
                fence_proxy_async();
                mbar_expect_tx(&sm.full_bar[my_slot], PIECE_BYTES);
                tma_load_1d(sm.ring[my_slot], key + (size_t)k2 * PIECE_CPLX, PIECE_BYTES, &sm.full_bar[my_slot]);
            }
        }
    };

    for (int i = 0; i < n_iters; ++i) {
        const uint32_t a = mod_switch(__ldg(lwe + i));                           // a == 0 is NOT skipped
        cta_sync();          // the accumulator polynomial is complete in the tile
        // ct1 = acc * X^a - acc and both signed digits: level 2 goes into the FFT registers now, level 1 waits as packed int16
        uint32_t d1pack[16];
#pragma unroll
        for (int m = 0; m < 16; ++m) {
            const int j = T + 256 * m;
            const uint32_t s0 = ((uint32_t)j - a) & (2 * N - 1), s1 = (s0 + M) & (2 * N - 1);
            uint64_t r0 = pb[s0 & (N - 1)], r1 = pb[s1 & (N - 1)];
            r0 = (s0 >= (uint32_t)N) ? (uint64_t)0 - r0 : r0;
            r1 = (s1 >= (uint32_t)N) ? (uint64_t)0 - r1 : r1;
            const uint64_t o0 = (uint64_t)__double_as_longlong(re[m]), o1 = (uint64_t)__double_as_longlong(im[m]);
            int a2, a1, b2, b1;
            signed_digits2(r0 - o0, base_log, a2, a1);
            signed_digits2(r1 - o1, base_log, b2, b1);
            re[m] = (double)a2; im[m] = (double)b2;
            d1pack[m] = ((uint32_t)a1 & 0xFFFFu) | ((uint32_t)b1 << 16);
        }
        double ore[16], oim[16];
#pragma unroll
        for (int g = 0; g < 16; ++g) { ore[g] = 0.0; oim[g] = 0.0; }

#pragma unroll
        for (int lvslot = 0; lvslot < LEVELS; ++lvslot) {
            if (lvslot == 1) {
#pragma unroll
                for (int m = 0; m < 16; ++m) {
                    re[m] = (double)(int)(short)(d1pack[m] & 0xFFFFu);
                    im[m] = (double)((int)d1pack[m] >> 16);
                }
            }
            Fft4096<TmemTw>::fwd(re, im, tile, twd, T, cta_sync);
            // my spectrum -> the partner's landing buffer, once the partner has released it (it read the previous one)
            if (use >= 1) wait_cluster(&sm.peer_free, (use - 1) & 1u);
#pragma unroll
            for (int g = 0; g < 16; ++g) st_async(peer_recv + (uint32_t)(g * THREADS * 16), re[g], im[g], peer_full);
            const int piece0 = (i * LEVELS + lvslot) * 2 * CHUNKS;
            mac_half(ore, oim, re, im, false, piece0);                            // own row, while the partner's spectrum is in flight
            if (!mbar_try_wait(&sm.recv_full, use & 1u)) mbar_wait(&sm.recv_full, use & 1u);
            if (T == 0) mbar_expect_tx(&sm.recv_full, SPEC_BYTES);                // re-armed: the partner sends again only after my release below
            mac_half(ore, oim, re, im, true, piece0 + CHUNKS);                    // partner row from the landing buffer
            cta_sync();                                                           // everybody has read the landing buffer
            if (T == 0) remote_arrive(peer_peer_free);                            // ... which the partner may now overwrite
            ++use;
        }
#pragma unroll
        for (int g = 0; g < 16; ++g) { re[g] = ore[g]; im[g] = oim[g]; }
        Fft4096<TmemTw>::inv(re, im, tile, twd, T, cta_sync);
        cta_sync();          // everybody is past its exchange reads: the tile becomes the accumulator polynomial again
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            uint32_t v[16];
            tmem_ld16(tmem_acc + 16 * kk, v);
            tmem_wait_ld();
#pragma unroll
            for (int mm = 0; mm < 4; ++mm) {
                const int m = 4 * kk + mm, j = T + 256 * m;
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
            tmem_st16(tmem_acc + 16 * kk, v);
        }
        tmem_wait_st();
    }

    // sample extraction of coefficient 0: out[0] = A[0], out[N - j] = -A[j]; body = B[0]
    if (many.fn) {
        const int nf = tbx::many_fn_count(many, lut_idx, ct);
        tbx::extract_many_regs<16, 256, N, 1>(out, out_slot[ct], nf, tbx::many_step(many, nf, N), w, T, re, im);
    } else {
        uint64_t *o = out + (size_t)(out_slot ? out_slot[ct] : ct) * (N + 1);
        if (w == 0) {
#pragma unroll
            for (int m = 0; m < 16; ++m) {
                const int j = T + 256 * m;
                const uint64_t v0 = (uint64_t)__double_as_longlong(re[m]), v1 = (uint64_t)__double_as_longlong(im[m]);
                if (j == 0) o[0] = v0; else o[N - j] = (uint64_t)0 - v0;
                o[N - (j + M)] = (uint64_t)0 - v1;
            }
        } else if (T == 0) {
            o[N] = (uint64_t)__double_as_longlong(re[0]);
        }
    }
    tc_fence_before();
    cluster_sync_all();      // nobody leaves while the partner could still address its shared memory
    if (W == 0) tmem_dealloc<512>(sm.tmem_base);
}

// std key [ggsw i][level L 0..1 = level 1, 2][row r][col c][N] -> the per-output-polynomial ring order
__global__ void __launch_bounds__(THREADS)
bsk_convert_n8192_kernel(const uint64_t *__restrict__ bsk_std, cplx *__restrict__ bskf, const cplx *__restrict__ tbl, int n_ggsw) {
    extern __shared__ __align__(16) unsigned char conv_smem[];
    cplx *tile = reinterpret_cast<cplx *>(conv_smem);
    const int qd = blockIdx.x, T = threadIdx.x;
    const int c = qd & 1, r = (qd >> 1) & 1, L = (qd >> 2) & 1, i = qd >> 3;
    const uint64_t *src = bsk_std + (size_t)qd * N;
    const double scale = 1.3234889800848443e-23;      // 2^-76 = 2^-64 (torus) / 4096 (inverse transform)
    double re[16], im[16];
#pragma unroll
    for (int m = 0; m < 16; ++m) {
        const int j = T + 256 * m;
        re[m] = DMUL((double)(long long)src[j], scale);
        im[m] = DMUL((double)(long long)src[j + M], scale);
    }
    Fft4096<GlobalTw>::fwd(re, im, tile, GlobalTw{tbl, T}, T, BlockSync{});
    const int lvslot = (L == 1) ? 0 : 1;               // std index L = level - 1; level 2 is consumed first
    const int sel = (r == c) ? 0 : 1;
#pragma unroll
    for (int g = 0; g < 16; ++g) {
        cplx v; v.x = re[g]; v.y = im[g];
        bskf[(key_piece(n_ggsw, c, i, lvslot, sel, g / QPP) * QPP + (g % QPP)) * THREADS + T] = v;
    }
}

}  // namespace tb8192

namespace tbk {

// signed_digits2 works on the top 32 bits of a word: base_log * LEVELS <= 31.  Larger bases (accepted up to B * l = 52) run on
// pbs_generic.cu, whose decomposition is 64-bit.
bool pbs_n8192_supported(int poly_size, int glwe_dim, int pbs_level, int pbs_base_log, int grouping_factor) {
    return poly_size == tb8192::N && glwe_dim == 1 && pbs_level == tb8192::LEVELS && pbs_base_log * tb8192::LEVELS <= 31 && grouping_factor == 0;
}

void pbs_n8192_make_table(double *t) { tb16x_make_table_8192(t); }

cudaError_t pbs_n8192_configure() {
    cudaError_t e = cudaFuncSetAttribute(tb8192::bsk_convert_n8192_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tb8192::TILE * 16);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(tb8192::pbs_n8192_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(tb8192::Smem));
}

cudaError_t launch_pbs_n8192(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskf, const void *tbl,
                             uint64_t *out, const uint32_t *out_slot, tbk::ManyLut many, int batch, int n, int base_log, int n_iters, int n_ggsw,
                             cudaStream_t stream) {
    if (batch <= 0) return cudaSuccess;
    tb8192::pbs_n8192_kernel<<<2 * batch, tb8192::THREADS, sizeof(tb8192::Smem), stream>>>(
        lwe_small, lut_idx, luts, reinterpret_cast<const tb::cplx *>(bskf), reinterpret_cast<const tb::cplx *>(tbl), out, out_slot, many, n, base_log,
        n_iters, n_ggsw);
    return cudaGetLastError();
}

cudaError_t launch_bsk_convert_n8192(const uint64_t *bsk_std, void *bskf, const void *tbl, int n_ggsw, cudaStream_t stream) {
    tb8192::bsk_convert_n8192_kernel<<<n_ggsw * 8, tb8192::THREADS, tb8192::TILE * 16, stream>>>(bsk_std, reinterpret_cast<tb::cplx *>(bskf),
                                                                               reinterpret_cast<const tb::cplx *>(tbl), n_ggsw);
    return cudaGetLastError();
}

}  // namespace tbk
