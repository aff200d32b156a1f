// pbs_generic.cu -- programmable bootstrap for every classic shortint parameter set the specialised kernels do not cover
// (SURVEY section 8(f) N4): polynomial sizes 256 ... 32768, GLWE dimension 1 ... 5, any number of PBS decomposition levels --
// PARAM_MESSAGE_1_CARRY_0 ... PARAM_MESSAGE_8_CARRY_0 (shortint/parameters/mod.rs:598-1136).  Same arithmetic as pbs_v4.cu, restated
// from bootstrap.rs:242-364 (blind rotation), ggsw.rs:477-598 (external product: levels l..1, rows, columns),
// math/decomposition.rs:25-86 + iter.rs:120-127 (multi-level signed decomposition with carry), fft/mod.rs:220-326 (fold/twist) and
// glwe_sample_extraction.rs:91-147, but with none of that kernel's shape assumptions:
//
//   * N <= 8192: one CTA per ciphertext, T = min(512, N/8) threads; the accumulator ((k+1) * N u64, <= 128 KiB) and ONE transform buffer
//     (N/2 complex, <= 64 KiB) live in shared memory;
//   * the size-N/2 complex FFT runs in place in that buffer, two radix-2 stages per pass in registers (forward DIF: natural ->
//     bit-reversed, inverse DIT: back), twiddles from per-pass shared tables, buffer slots XOR-swizzled so that no pass has bank
//     conflicts; nothing is ever reordered -- the Fourier key is produced by the same device function and multiplied position by position;
//   * every thread keeps the Fourier-domain output of "its" PER = (N/2)/T positions for all k+1 output polynomials in registers
//     (<= 16 complex values), so the (k+1)(level) forward transforms of an iteration share the one buffer;
//   * the Fourier key [ggsw][level][row][col][N/2] is read with coalesced 16-byte loads, once per ciphertext and iteration.
//
//   * multi-bit PBS (grouping factor 2, 3; N <= 8192) combines the group's GGSWs on the fly in the Fourier domain (GF template parameter);
//   * N = 16384, 32768: second kernel further down (working set in an L2-resident scratch area).
//
// This is the coverage kernel, not the tuned one: N = 2048, k = 1, one level stays on pbs_v4.cu / pbs_v8.cu (TFHE_B200_PBS_KERNEL=generic
// forces this one for cross-checks).  Measured 2.4 ... 6.1 TFLOP/s algorithmic against 15.8 for the tuned kernels (DESIGN.md K12).
#include "kernels.h"
#include "sample_extract.cuh"
#include <type_traits>
#include "fft_core.cuh"
#include "pbs16_common.cuh"      // Tensor Memory helpers (tcgen05.alloc / ld / st)

namespace tbg {
using tb::cplx;

template <int LOGN, int K1 = 0>
struct Shape {
    static constexpr int N = 1 << LOGN, M = N / 2;
    static constexpr bool R8 = K1 == 2 && M >= 1024;          // k = 1: three stages per FFT pass (Fft8), 8 positions per thread
    static constexpr int PER = R8 ? 8 : M > 2048 ? M / 512 : 4;   // otherwise one radix-4 butterfly per thread and pass (two above N = 4096)
    static constexpr int T = M / PER;
    // N = 4096, 8192 with 8 positions per thread: the 16 complex Fourier accumulators of a thread (64 registers) are parked in its Tensor
    // Memory lane while the FFT passes run (ncu on N = 8192: 1.0 G spill instructions, and with 208 KiB of shared memory there is no L1
    // left, so every spill reload was an L2 round trip -- long_scoreboard 3.1 of 12.5 cycles per instruction)
    static constexpr bool TM = R8 && M >= 2048;
    static constexpr int TM_SLOT = 128;                       // columns per warp: 64 accumulator + 32 twist factors (+ 32 unused)
    static constexpr int TM_COLS = T / 128 * TM_SLOT;         // warps sharing a lane quarter x slot
    // resident CTAs per SM the register allocation must allow: N = 4096 two 512-thread CTAs (64 registers); N = 512 ... 2048 are capped
    // at 128 registers, which doubles their occupancy (ncu: 234 registers, 8 warps per SM, latency bound; +2 ... +18 %).  N = 256 (k = 5,
    // 24 complex accumulators per thread) is faster uncapped (measured: 80.7 k vs 56.7 k KS-PBS/s with a 168-register cap)
    static constexpr int MINB = M == 2048 ? 2 : M == 1024 ? 2 : M == 512 ? 4 : M == 256 ? 8 : 1;
};

__device__ __forceinline__ cplx cmul(cplx a, cplx b) {
    cplx r;
    r.x = DFMA(a.x, b.x, -DMUL(a.y, b.y));
    r.y = DFMA(a.x, b.y, DMUL(a.y, b.x));
    return r;
}
__device__ __forceinline__ cplx cmul_conj(cplx a, cplx b) {   // a * conj(b)
    cplx r;
    r.x = DFMA(a.x, b.x, DMUL(a.y, b.y));
    r.y = DFMA(a.y, b.x, -DMUL(a.x, b.y));
    return r;
}

// W_M^e = exp(-2*pi*i*e/M), e < M/2, from the twist table tw[j] = exp(i*pi*j/N), j < M (N = 2M): W_M^e = conj(tw[4e]) for e < M/4,
// and -i * conj(tw[4e - M]) above
template <int M>
__device__ __forceinline__ cplx root(const cplx *__restrict__ tw, int e) {
    if (M < 4) { cplx r; r.x = e ? 0.0 : 1.0; r.y = e ? -1.0 : 0.0; return r; }
    const bool hi = e >= M / 4;
    const cplx t = __ldg(tw + (hi ? 4 * e - M : 4 * e));
    cplx r;
    r.x = hi ? -t.y : t.x;
    r.y = hi ? -t.x : -t.y;
    return r;
}

// Shared-memory tables of one transform size M: wt = the radix-4 passes' first-stage twiddles W_{4q}^j (j < q) for q = 1, 4, 16, ...,
// stored pass by pass (offset (q - 1) / 3) so that consecutive threads read consecutive entries; the second-stage twiddle is its
// square.  When log2 M is odd one plain radix-2 stage remains, with W_M^b from rt[e] = W_M^e, e < M/4 (the upper half by symmetry).
template <int M> struct Log2 { static constexpr int v = 1 + Log2<M / 2>::v; };
template <> struct Log2<1> { static constexpr int v = 0; };
template <int M>
struct Tables {
    static constexpr bool ODD = (Log2<M>::v & 1) != 0;
    static constexpr int QMAX = ODD ? M / 8 : M / 4;
    static constexpr int WT = (4 * QMAX - 1) / 3;
    static constexpr int RT = ODD ? M / 4 : 0;
    static constexpr int ENTRIES = WT + RT;
};

// tw[t] = exp(i*pi*t/N) with N = n_over_m * M: W_{4q}^j = conj(tw[j * N / (2q)]), W_M^e = conj(tw[2 * e * N / M])
template <int M, int T>
__device__ __forceinline__ void make_tables(cplx *tbl, const cplx *__restrict__ tw, int n_over_m) {
    for (int q = 1; q <= Tables<M>::QMAX; q <<= 2)
        for (int j = threadIdx.x; j < q; j += T) {
            const cplx w = __ldg(tw + (size_t)j * (n_over_m * M / (2 * q)));
            cplx r; r.x = w.x; r.y = -w.y;
            tbl[(q - 1) / 3 + j] = r;
        }
    if (Tables<M>::ODD)
        for (int e = threadIdx.x; e < M / 4; e += T) {
            const cplx w = __ldg(tw + (size_t)e * 2 * n_over_m);
            cplx r; r.x = w.x; r.y = -w.y;
            tbl[Tables<M>::WT + e] = r;
        }
}

template <int M>
__device__ __forceinline__ cplx sroot(const cplx *tbl, int e) {      // W_M^e, e < M/2, for the radix-2 stage
    const bool hi = e >= M / 4;
    const cplx t = tbl[Tables<M>::WT + (hi ? e - M / 4 : e)];
    cplx r;
    r.x = hi ? t.y : t.x;          // (-i) * (x + iy) = y - ix
    r.y = hi ? -t.x : t.y;
    return r;
}
__device__ __forceinline__ cplx cadd(cplx a, cplx b) { cplx r; r.x = DADD(a.x, b.x); r.y = DADD(a.y, b.y); return r; }
__device__ __forceinline__ cplx csub(cplx a, cplx b) { cplx r; r.x = DSUB(a.x, b.x); r.y = DSUB(a.y, b.y); return r; }
__device__ __forceinline__ cplx mul_neg_i(cplx a) { cplx r; r.x = a.y; r.y = -a.x; return r; }
__device__ __forceinline__ cplx mul_pos_i(cplx a) { cplx r; r.x = -a.y; r.y = a.x; return r; }
__device__ __forceinline__ cplx csqr(cplx a) { cplx r; r.x = DFMA(a.x, a.x, -DMUL(a.y, a.y)); r.y = DMUL(DADD(a.x, a.x), a.y); return r; }

// Element i of a transform buffer lives at slot SW(i): the low three slot bits are XOR-ed with bits 3-4 of i, which makes the
// 16-byte accesses of every pass conflict free -- consecutive elements (q >= 8), the q = 4 pass (elements 16 g + j + 4 m) and the
// q = 1 pass (elements 4 b + m) each spread a quarter-warp over all eight 16-byte bank groups.
__device__ __forceinline__ int SW(int i) { return i ^ ((i >> 3) & 3) ^ ((i >> 2) & 4); }

// forward: natural order in, bit-reversed positions out (radix-2 DIF stages taken two at a time).  Ends with a barrier.
template <int M, int T>
__device__ __forceinline__ void fft_fwd(cplx *buf, const cplx *tbl) {
    int half = M / 2;
    if (Tables<M>::ODD) {                      // odd stage count: one plain radix-2 stage first
        __syncthreads();
        for (int b = threadIdx.x; b < M / 2; b += T) {
            const cplx u = buf[SW(b)], v = buf[SW(b + M / 2)];
            buf[SW(b)] = cadd(u, v);
            buf[SW(b + M / 2)] = cmul(csub(u, v), sroot<M>(tbl, b));
        }
        half >>= 1;
    }
    for (; half >= 2; half >>= 2) {            // stages `half` and `half / 2` in registers
        __syncthreads();
        const int q = half >> 1;
        const cplx *wq = tbl + (q - 1) / 3;
        for (int b = threadIdx.x; b < M / 4; b += T) {
            const int j = b & (q - 1), i0 = ((b - j) << 2) + j;
            const int p0 = SW(i0), p1 = SW(i0 + q), p2 = SW(i0 + 2 * q), p3 = SW(i0 + 3 * q);
            const cplx a0 = buf[p0], a1 = buf[p1], a2 = buf[p2], a3 = buf[p3];
            const cplx b0 = cadd(a0, a2), b1 = cadd(a1, a3);
            const cplx b2 = csub(a0, a2), b3 = mul_neg_i(csub(a1, a3));
            cplx c1 = csub(b0, b1), c2 = cadd(b2, b3), c3 = csub(b2, b3);
            if (q > 1) {
                const cplx w1 = wq[j], w2 = csqr(w1);
                c1 = cmul(c1, w2);
                c2 = cmul(c2, w1);             // both halves of the first stage carry W_{4q}^j ...
                c3 = cmul(cmul(c3, w1), w2);   // ... and the lower pair also the second stage's W_{2q}^j
            }
            buf[p0] = cadd(b0, b1);
            buf[p1] = c1;
            buf[p2] = c2;
            buf[p3] = c3;
        }
    }
    __syncthreads();
}

// inverse (unscaled): bit-reversed positions in, natural order out.  Ends with a barrier.
template <int M, int T>
__device__ __forceinline__ void fft_inv(cplx *buf, const cplx *tbl) {
    for (int q = 1; 4 * q <= M; q <<= 2) {     // stages `q` and `2q`
        __syncthreads();
        const cplx *wq = tbl + (q - 1) / 3;
        for (int b = threadIdx.x; b < M / 4; b += T) {
            const int j = b & (q - 1), i0 = ((b - j) << 2) + j;
            const int p0 = SW(i0), p1 = SW(i0 + q), p2 = SW(i0 + 2 * q), p3 = SW(i0 + 3 * q);
            cplx c0 = buf[p0], c1 = buf[p1], c2 = buf[p2], c3 = buf[p3];
            if (q > 1) {
                const cplx w1 = wq[j], w2 = csqr(w1);
                c1 = cmul_conj(c1, w2);
                c2 = cmul_conj(c2, w1);
                c3 = cmul_conj(cmul_conj(c3, w1), w2);
            }
            const cplx b0 = cadd(c0, c1), b1 = csub(c0, c1), b2 = cadd(c2, c3), b3 = mul_pos_i(csub(c2, c3));
            buf[p0] = cadd(b0, b2);
            buf[p2] = csub(b0, b2);
            buf[p1] = cadd(b1, b3);
            buf[p3] = csub(b1, b3);
        }
    }
    if (Tables<M>::ODD) {
        __syncthreads();
        for (int b = threadIdx.x; b < M / 2; b += T) {
            const cplx u = buf[SW(b)], v = cmul_conj(buf[SW(b + M / 2)], sroot<M>(tbl, b));
            buf[SW(b)] = cadd(u, v);
            buf[SW(b + M / 2)] = csub(u, v);
        }
    }
    __syncthreads();
}

// ---- the same transform with THREE radix-2 stages per shared-memory pass (8 points per thread) -----------------------------------
// used where a thread's registers allow it (k = 1: 16 complex Fourier accumulators + 8 points): 4 passes instead of 6 at N = 4096 and
// 8192.  log2(M) mod 3 leftover stages run first (one radix-2 or one radix-4 pass over the whole buffer), then passes with q = M'/8,
// M'/64, ..., 1.  Inside a pass the stage twiddles W_{8q}^j, W_{4q}^j, W_{2q}^j are powers of w1 = W_{8q}^j and commute with the later
// butterflies of their half, so they are applied once at the end as w1^brev3(a) on register a; only the constants W_8^r, W_4^r sit
// between the stages.  Slot swizzle: low three bits XOR bits 3-5 (conflict free for consecutive elements, q = 8 and q = 1).
constexpr double kInvSqrt2 = 0.70710678118654752440;

template <int M, int T>
struct Fft8 {
    static constexpr int R = Log2<M>::v % 3;
    static constexpr int MP = M >> R;              // size of the sub-transforms the radix-8 passes see
    static constexpr int QMAX = MP / 8;
    static constexpr int W8 = (8 * QMAX - 1) / 7;  // pass q = 8^i at offset (q - 1) / 7
    static constexpr int LEFT = R == 0 ? 0 : M / 4;
    static constexpr int ENTRIES = W8 + LEFT;
    __device__ static __forceinline__ int sw(int i) { return i ^ ((i >> 3) & 7); }

    __device__ static __forceinline__ void make(cplx *tbl, const cplx *__restrict__ tw, int n_over_m) {
        for (int q = 1; q <= QMAX; q <<= 3)
            for (int j = threadIdx.x; j < q; j += T) {
                const cplx w = __ldg(tw + (size_t)j * (n_over_m * M / (4 * q)));      // W_{8q}^j = conj(tw[j N / (4q)])
                cplx r; r.x = w.x; r.y = -w.y;
                tbl[(q - 1) / 7 + j] = r;
            }
        if (R != 0)
            for (int e = threadIdx.x; e < M / 4; e += T) {
                const cplx w = __ldg(tw + (size_t)e * 2 * n_over_m);                  // W_M^e
                cplx r; r.x = w.x; r.y = -w.y;
                tbl[W8 + e] = r;
            }
    }
    __device__ static __forceinline__ cplx left_root(const cplx *tbl, int e) {        // W_M^e, e < M/2
        const bool hi = e >= M / 4;
        const cplx t = tbl[W8 + (hi ? e - M / 4 : e)];
        cplx r;
        r.x = hi ? t.y : t.x;
        r.y = hi ? -t.x : t.y;
        return r;
    }

    __device__ static __forceinline__ void fwd(cplx *buf, const cplx *tbl) {
        if (R == 1) {
            __syncthreads();
            for (int b = threadIdx.x; b < M / 2; b += T) {
                const cplx u = buf[sw(b)], v = buf[sw(b + M / 2)];
                buf[sw(b)] = cadd(u, v);
                buf[sw(b + M / 2)] = cmul(csub(u, v), left_root(tbl, b));
            }
        } else if (R == 2) {
            __syncthreads();
            constexpr int q = M / 4;
            for (int b = threadIdx.x; b < M / 4; b += T) {
                const int p0 = sw(b), p1 = sw(b + q), p2 = sw(b + 2 * q), p3 = sw(b + 3 * q);
                const cplx a0 = buf[p0], a1 = buf[p1], a2 = buf[p2], a3 = buf[p3];
                const cplx b0 = cadd(a0, a2), b1 = cadd(a1, a3), b2 = csub(a0, a2), b3 = mul_neg_i(csub(a1, a3));
                const cplx w1 = tbl[W8 + b], w2 = csqr(w1);
                buf[p0] = cadd(b0, b1);
                buf[p1] = cmul(csub(b0, b1), w2);
                buf[p2] = cmul(cadd(b2, b3), w1);
                buf[p3] = cmul(cmul(csub(b2, b3), w1), w2);
            }
        }
        for (int q = QMAX; q >= 1; q >>= 3) {
            __syncthreads();
            const cplx *wq = tbl + (q - 1) / 7;
            for (int b = threadIdx.x; b < M / 8; b += T) {
                const int j = b & (q - 1), i0 = ((b - j) << 3) + j;
                cplx x[8];
#pragma unroll
                for (int m = 0; m < 8; ++m) x[m] = buf[sw(i0 + m * q)];
                // stage A: pairs (a, a + 4), constants W_8^a
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    const cplx u = x[a], d = csub(x[a], x[a + 4]);
                    x[a] = cadd(u, x[a + 4]);
                    cplx r;
                    if (a == 0) r = d;
                    else if (a == 1) { r.x = DMUL(DADD(d.x, d.y), kInvSqrt2); r.y = DMUL(DSUB(d.y, d.x), kInvSqrt2); }
                    else if (a == 2) r = mul_neg_i(d);
                    else { r.x = DMUL(DSUB(d.y, d.x), kInvSqrt2); r.y = -DMUL(DADD(d.x, d.y), kInvSqrt2); }
                    x[a + 4] = r;
                }
                // stage B: pairs (a, a + 2) inside each half, constants W_4^a
#pragma unroll
                for (int base = 0; base < 8; base += 4) {
                    const cplx u0 = x[base], u1 = x[base + 1];
                    const cplx d0 = csub(u0, x[base + 2]), d1 = mul_neg_i(csub(u1, x[base + 3]));
                    x[base] = cadd(u0, x[base + 2]);
                    x[base + 1] = cadd(u1, x[base + 3]);
                    x[base + 2] = d0;
                    x[base + 3] = d1;
                }
                // stage C: pairs (a, a + 1)
#pragma unroll
                for (int base = 0; base < 8; base += 2) {
                    const cplx u = x[base], v = x[base + 1];
                    x[base] = cadd(u, v);
                    x[base + 1] = csub(u, v);
                }
                if (q > 1) {                       // register a carries w1^brev3(a): a = 4 -> 1, 2 -> 2, 6 -> 3, 1 -> 4, 5 -> 5, 3 -> 6, 7 -> 7
                    const cplx w1 = wq[j], w2 = csqr(w1), w3 = cmul(w1, w2), w4 = csqr(w2);
                    x[4] = cmul(x[4], w1);
                    x[2] = cmul(x[2], w2);
                    x[6] = cmul(x[6], w3);
                    x[1] = cmul(x[1], w4);
                    x[5] = cmul(x[5], cmul(w4, w1));
                    x[3] = cmul(x[3], cmul(w4, w2));
                    x[7] = cmul(x[7], cmul(w4, w3));
                }
#pragma unroll
                for (int m = 0; m < 8; ++m) buf[sw(i0 + m * q)] = x[m];
            }
        }
        __syncthreads();
    }

    __device__ static __forceinline__ void inv(cplx *buf, const cplx *tbl) {
        for (int q = 1; q <= QMAX; q <<= 3) {
            __syncthreads();
            const cplx *wq = tbl + (q - 1) / 7;
            for (int b = threadIdx.x; b < M / 8; b += T) {
                const int j = b & (q - 1), i0 = ((b - j) << 3) + j;
                cplx x[8];
#pragma unroll
                for (int m = 0; m < 8; ++m) x[m] = buf[sw(i0 + m * q)];
                if (q > 1) {
                    const cplx w1 = wq[j], w2 = csqr(w1), w3 = cmul(w1, w2), w4 = csqr(w2);
                    x[4] = cmul_conj(x[4], w1);
                    x[2] = cmul_conj(x[2], w2);
                    x[6] = cmul_conj(x[6], w3);
                    x[1] = cmul_conj(x[1], w4);
                    x[5] = cmul_conj(x[5], cmul(w4, w1));
                    x[3] = cmul_conj(x[3], cmul(w4, w2));
                    x[7] = cmul_conj(x[7], cmul(w4, w3));
                }
#pragma unroll
                for (int base = 0; base < 8; base += 2) {
                    const cplx u = x[base], v = x[base + 1];
                    x[base] = cadd(u, v);
                    x[base + 1] = csub(u, v);
                }
#pragma unroll
                for (int base = 0; base < 8; base += 4) {
                    const cplx u0 = x[base], u1 = x[base + 1], v0 = x[base + 2], v1 = mul_pos_i(x[base + 3]);
                    x[base] = cadd(u0, v0);
                    x[base + 2] = csub(u0, v0);
                    x[base + 1] = cadd(u1, v1);
                    x[base + 3] = csub(u1, v1);
                }
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    const cplx u = x[a], d = x[a + 4];
                    cplx v;                        // d * conj(W_8^a)
                    if (a == 0) v = d;
                    else if (a == 1) { v.x = DMUL(DSUB(d.x, d.y), kInvSqrt2); v.y = DMUL(DADD(d.x, d.y), kInvSqrt2); }
                    else if (a == 2) v = mul_pos_i(d);
                    else { v.x = -DMUL(DADD(d.x, d.y), kInvSqrt2); v.y = DMUL(DSUB(d.x, d.y), kInvSqrt2); }
                    x[a] = cadd(u, v);
                    x[a + 4] = csub(u, v);
                }
#pragma unroll
                for (int m = 0; m < 8; ++m) buf[sw(i0 + m * q)] = x[m];
            }
        }
        if (R == 1) {
            __syncthreads();
            for (int b = threadIdx.x; b < M / 2; b += T) {
                const cplx u = buf[sw(b)], v = cmul_conj(buf[sw(b + M / 2)], left_root(tbl, b));
                buf[sw(b)] = cadd(u, v);
                buf[sw(b + M / 2)] = csub(u, v);
            }
        } else if (R == 2) {
            __syncthreads();
            constexpr int q = M / 4;
            for (int b = threadIdx.x; b < M / 4; b += T) {
                const int p0 = sw(b), p1 = sw(b + q), p2 = sw(b + 2 * q), p3 = sw(b + 3 * q);
                const cplx w1 = tbl[W8 + b], w2 = csqr(w1);
                const cplx c0 = buf[p0], c1 = cmul_conj(buf[p1], w2), c2 = cmul_conj(buf[p2], w1), c3 = cmul_conj(cmul_conj(buf[p3], w1), w2);
                const cplx b0 = cadd(c0, c1), b1 = csub(c0, c1), b2 = cadd(c2, c3), b3 = mul_pos_i(csub(c2, c3));
                buf[p0] = cadd(b0, b2);
                buf[p2] = csub(b0, b2);
                buf[p1] = cadd(b1, b3);
                buf[p3] = csub(b1, b3);
            }
        }
        __syncthreads();
    }
};

// the two-stages-per-pass transform behind the same interface
template <int M, int T>
struct Fft4 {
    static constexpr int ENTRIES = Tables<M>::ENTRIES;
    __device__ static __forceinline__ int sw(int i) { return SW(i); }
    __device__ static __forceinline__ void make(cplx *tbl, const cplx *__restrict__ tw, int n_over_m) { make_tables<M, T>(tbl, tw, n_over_m); }
    __device__ static __forceinline__ void fwd(cplx *buf, const cplx *tbl) { fft_fwd<M, T>(buf, tbl); }
    __device__ static __forceinline__ void inv(cplx *buf, const cplx *tbl) { fft_inv<M, T>(buf, tbl); }
};

// digit of level `lv` (1 = most significant) of the `levels`-level signed decomposition of x: closest representable
// (decomposer.rs:98-118), then the carry chain from the least significant level up (iter.rs:120-127)
__device__ __forceinline__ int64_t signed_digit(uint64_t x, int base_log, int levels, int lv) {
    const int shift = 64 - base_log * levels - 1;
    uint64_t state = (((x >> shift) + 1) & ~(uint64_t)1) >> 1;      // closest_representable(x) >> (64 - base_log * levels)
    const uint64_t mask = ((uint64_t)1 << base_log) - 1;
    uint64_t digit = 0;
    for (int l = levels; l >= lv; --l) {
        digit = state & mask;
        state >>= base_log;
        const uint64_t carry = (((digit - 1) | state) & digit) >> (base_log - 1);
        state += carry;
        digit -= carry << base_log;
    }
    return (int64_t)digit;
}

// a thread's K1 x PER complex accumulators in its own Tensor Memory lane (4 columns per value)
template <int K1, int PER>
struct TmemAcc {
    uint32_t base;
    __device__ __forceinline__ void store(const cplx (&o)[K1][PER]) const {
#pragma unroll
        for (int k = 0; k < K1 * PER / 4; ++k) {
            uint32_t v[16];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const cplx z = o[(4 * k + e) / PER][(4 * k + e) % PER];
                v[4 * e] = (uint32_t)__double2loint(z.x); v[4 * e + 1] = (uint32_t)__double2hiint(z.x);
                v[4 * e + 2] = (uint32_t)__double2loint(z.y); v[4 * e + 3] = (uint32_t)__double2hiint(z.y);
            }
            tb16k::tmem_st16(base + 16 * k, v);
        }
        tb16k::tmem_wait_st();
    }
    __device__ __forceinline__ void load_col(int c, cplx (&oc)[PER]) const {
#pragma unroll
        for (int k = 0; k < PER / 4; ++k) {
            uint32_t v[16];
            tb16k::tmem_ld16(base + (uint32_t)(c * PER * 4 + 16 * k), v);
            tb16k::tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                oc[4 * k + e].x = __hiloint2double((int)v[4 * e + 1], (int)v[4 * e]);
                oc[4 * k + e].y = __hiloint2double((int)v[4 * e + 3], (int)v[4 * e + 2]);
            }
        }
    }
    __device__ __forceinline__ void load(cplx (&o)[K1][PER]) const {
#pragma unroll
        for (int c = 0; c < K1; ++c) load_col(c, o[c]);
    }
};

// w^e = exp(i*pi*e/N) for e in [0, 2N) from the twist table (e < N/2) and the quadrant
template <int N>
__device__ __forceinline__ cplx root2n(const cplx *__restrict__ tw, uint32_t e) {
    const cplx t = __ldg(tw + (e & (N / 2 - 1)));
    const uint32_t quad = (e / (N / 2)) & 3u;
    cplx r;
    r.x = quad == 0 ? t.x : quad == 1 ? -t.y : quad == 2 ? -t.x : t.y;
    r.y = quad == 0 ? t.y : quad == 1 ? t.x : quad == 2 ? -t.y : -t.x;
    return r;
}

// GF = 0: classic blind rotation.  GF = 2, 3: multi-bit (lwe_multi_bit_programmable_bootstrapping.rs:18-84,295-546, deterministic order):
// per group of GF mask elements acc <- G (x) acc with G = G_0 + sum_j G_j * X^(deg_j) combined on the fly in the Fourier domain -- position
// `pos` of the transform holds the evaluation at zeta = w^(1 - 4*brev(pos)), so the monomial's spectrum there is w^(deg_j * (1 - 4*brev(pos)))
// (fft/mod.rs:408-445).  n_iters counts groups.
template <int LOGN, int K1, int GF>
__global__ void __launch_bounds__(Shape<LOGN, K1>::T, Shape<LOGN, K1>::MINB)
pbs_generic_kernel(const uint64_t *__restrict__ lwe_small, const uint32_t *__restrict__ lut_idx, const uint64_t *__restrict__ luts,
                   const cplx *__restrict__ bskf, const cplx *__restrict__ tw, uint64_t *__restrict__ out,
                   const uint32_t *__restrict__ out_slot, const tbk::ManyLut many, int n, int base_log, int levels, int n_iters) {
    using S = Shape<LOGN, K1>;
    constexpr int N = S::N, M = S::M, PER = S::PER, T = S::T;
    using F = typename std::conditional<S::R8, Fft8<M, T>, Fft4<M, T>>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *acc = reinterpret_cast<uint64_t *>(smem_raw);                 // [K1][N]
    cplx *buf = reinterpret_cast<cplx *>(smem_raw + (size_t)K1 * N * 8);      // [M]
    cplx *rt = buf + M;                                                       // [F::ENTRIES] twiddle tables
    const int ct = blockIdx.x, t = threadIdx.x;
    F::make(rt, tw, 2);
    constexpr bool TM = S::TM;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(rt + F::ENTRIES);
    TmemAcc<K1, PER> tacc{0};
    if (TM) {
        if (t < 32) tb16k::tmem_alloc<S::TM_COLS>(tmem_slot);
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        tacc.base = *tmem_slot + ((uint32_t)(((t >> 5) & 3) * 32) << 16) + (uint32_t)((t >> 7) * S::TM_SLOT);    // lane quarter = warp id % 4
        // the twist factors of this thread's positions never change: keep them in its Tensor Memory lane as well (ncu: with no L1 left
        // beside the shared memory, every __ldg(tw + j) of the fold / unfold steps waited for L2)
        cplx twv[1][PER];
#pragma unroll
        for (int q = 0; q < PER; ++q) twv[0][q] = __ldg(tw + t + T * q);
        TmemAcc<1, PER>{tacc.base + K1 * PER * 4}.store(twv);
    }
    const TmemAcc<1, PER> ttw{tacc.base + K1 * PER * 4};
    const uint64_t *lwe = lwe_small + (size_t)ct * (n + 1);
    const auto mod_switch = [](uint64_t x) { return (uint32_t)(((x >> (64 - LOGN - 2)) + 1) >> 1) & (2 * N - 1); };

    // acc <- LUT * X^(-b_hat)   (bootstrap.rs:262-270; polynomial_algorithms.rs:315-366)
    {
        const uint32_t a0 = (2 * N - mod_switch(__ldg(lwe + n))) & (2 * N - 1);
        const uint64_t *lut = luts + (size_t)(lut_idx ? lut_idx[ct] : 0) * K1 * N;
        for (int c = 0; c < K1; ++c)
            for (int j = t; j < N; j += T) {
                const uint32_t s = ((uint32_t)j - a0) & (2 * N - 1);
                const uint64_t v = __ldg(lut + c * N + (s & (N - 1)));
                acc[c * N + j] = s >= (uint32_t)N ? (uint64_t)0 - v : v;
            }
    }
    __syncthreads();

    for (int i = 0; i < n_iters; ++i) {
        uint32_t a_hat = 0;
        uint32_t deg[GF ? (1 << GF) : 1];                                    // multi-bit: monomial degree of GGSW j (:44-62)
        if (GF == 0) {
            a_hat = mod_switch(__ldg(lwe + i));
            if (a_hat == 0) continue;                                        // bootstrap.rs:281 (result-neutral)
        } else {
#pragma unroll
            for (int j = 1; j < (1 << GF); ++j) {
                uint64_t sum = 0;
#pragma unroll
                for (int mi = 0; mi < GF; ++mi)
                    if ((j >> (GF - 1 - mi)) & 1) sum += __ldg(lwe + GF * i + mi);
                deg[j] = mod_switch(sum);
            }
        }
        cplx o[K1][PER];
        if (!S::TM) {
#pragma unroll
            for (int c = 0; c < K1; ++c)
#pragma unroll
                for (int q = 0; q < PER; ++q) { o[c][q].x = 0.0; o[c][q].y = 0.0; }
        }
        const size_t ggsw_len = (size_t)levels * K1 * K1 * M;
        const cplx *ggsw = bskf + (size_t)i * (GF ? (1 << GF) : 1) * ggsw_len;
        bool parked = false;                                                 // TM: the accumulators are in Tensor Memory

        for (int lv = levels; lv >= 1; --lv) {                               // ggsw.rs:524: level l first
            for (int r = 0; r < K1; ++r) {
                // digits of (acc * X^a_hat - acc)[r] (bootstrap.rs:286-300; multi-bit: of acc[r] itself), folded (coefficient j +
                // i * coefficient j+M) and twisted
                const uint64_t *src = acc + r * N;
                cplx twq[PER];
                if (TM) ttw.load_col(0, twq);
#pragma unroll
                for (int q = 0; q < PER; ++q) {
                    const int j = t + T * q;
                    uint64_t v0, v1;
                    if (GF == 0) {
                        const uint32_t s0 = ((uint32_t)j - a_hat) & (2 * N - 1), s1 = ((uint32_t)(j + M) - a_hat) & (2 * N - 1);
                        v0 = src[s0 & (N - 1)]; v1 = src[s1 & (N - 1)];
                        v0 = (s0 >= (uint32_t)N ? (uint64_t)0 - v0 : v0) - src[j];
                        v1 = (s1 >= (uint32_t)N ? (uint64_t)0 - v1 : v1) - src[j + M];
                    } else {
                        v0 = src[j]; v1 = src[j + M];
                    }
                    cplx z;
                    z.x = (double)signed_digit(v0, base_log, levels, lv);
                    z.y = (double)signed_digit(v1, base_log, levels, lv);
                    buf[F::sw(j)] = cmul(z, TM ? twq[q] : __ldg(tw + j));
                }
                const cplx *g = ggsw + ((size_t)(lv - 1) * K1 + r) * K1 * M;
                if (TM && GF == 0 && LOGN >= 13) {                           // the key values this thread multiplies by after the transform: pull
#pragma unroll                                                               // them into L2 while the FFT passes run (no registers held).  N = 8192
                    // only: its key (453 MB) streams from HBM (3_3 +2.5 %); keys that fit the L2 lose 1.5 % to the extra instructions
                    for (int q = 0; q < PER; ++q)
#pragma unroll
                        for (int c = 0; c < K1; ++c) asm volatile("prefetch.global.L2 [%0];" ::"l"(g + (size_t)c * M + t + T * q));
                }
                F::fwd(buf, rt);
                if (TM) {                                                    // the accumulators live in registers only across this loop
                    if (parked) tacc.load(o);
                    else {
#pragma unroll
                        for (int c = 0; c < K1; ++c)
#pragma unroll
                            for (int q = 0; q < PER; ++q) { o[c][q].x = 0.0; o[c][q].y = 0.0; }
                    }
                }
#pragma unroll
                for (int q = 0; q < PER; ++q) {
                    const int pos = t + T * q;
                    const cplx f = buf[F::sw(pos)];
                    if (GF == 0) {
#pragma unroll
                        for (int c = 0; c < K1; ++c) {
                            const cplx gv = __ldg(g + (size_t)c * M + pos);
                            o[c][q].x = DFMA(f.x, gv.x, DFMA(-f.y, gv.y, o[c][q].x));
                            o[c][q].y = DFMA(f.x, gv.y, DFMA(f.y, gv.x, o[c][q].y));
                        }
                    } else {
                        // F * (G_0 + sum_j G_j * M_j) = F * G_0 + sum_j (F * M_j) * G_j
                        const uint32_t rot = (1u - 4u * (__brev((uint32_t)pos) >> (33 - LOGN))) & (2 * N - 1);
#pragma unroll
                        for (int j = 0; j < (1 << GF); ++j) {
                            const cplx fm = j == 0 ? f : cmul(f, root2n<N>(tw, (deg[j] * rot) & (2 * N - 1)));
#pragma unroll
                            for (int c = 0; c < K1; ++c) {
                                const cplx gv = __ldg(g + (size_t)j * ggsw_len + (size_t)c * M + pos);
                                o[c][q].x = DFMA(fm.x, gv.x, DFMA(-fm.y, gv.y, o[c][q].x));
                                o[c][q].y = DFMA(fm.x, gv.y, DFMA(fm.y, gv.x, o[c][q].y));
                            }
                        }
                    }
                }
                if (TM) { tacc.store(o); parked = true; }
                __syncthreads();                                             // the buffer is rewritten next
            }
        }
        // ct0[c] += round(inverse transform)   (fft/mod.rs:285-326; the 1/(N/2) and the 2^-64 of the key are folded into the key)
#pragma unroll
        for (int c = 0; c < K1; ++c) {
#pragma unroll
            if (TM) tacc.load_col(c, o[c]);
#pragma unroll
            for (int q = 0; q < PER; ++q) buf[F::sw(t + T * q)] = o[c][q];
            F::inv(buf, rt);
            cplx twq[PER];
            if (TM) ttw.load_col(0, twq);
#pragma unroll
            for (int q = 0; q < PER; ++q) {
                const int j = t + T * q;
                const cplx z = cmul_conj(buf[F::sw(j)], TM ? twq[q] : __ldg(tw + j));
                if (GF == 0) {
                    acc[c * N + j] += tb::from_torus_f64(z.x);
                    acc[c * N + j + M] += tb::from_torus_f64(z.y);
                } else {                                                     // dst = 0; dst += G (x) src (:503)
                    acc[c * N + j] = tb::from_torus_f64(z.x);
                    acc[c * N + j + M] = tb::from_torus_f64(z.y);
                }
            }
            __syncthreads();
        }
    }

    // sample extraction of coefficient 0 (glwe_sample_extraction.rs:91-147)
    if (many.fn) {
        const int nf = tbx::many_fn_count(many, lut_idx, ct);
        tbx::extract_many_acc(out, out_slot[ct], nf, tbx::many_step(many, nf, N), acc, N, K1 - 1, t, T);
    } else {
        uint64_t *dst = out + (size_t)(out_slot ? out_slot[ct] : ct) * ((size_t)(K1 - 1) * N + 1);
        for (int r = 0; r < K1 - 1; ++r)
            for (int j = t; j < N; j += T) dst[r * N + j] = j == 0 ? acc[r * N] : (uint64_t)0 - acc[r * N + N - j];
        if (t == 0) dst[(K1 - 1) * N] = acc[(K1 - 1) * N];
    }
    if (TM) {
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (t < 32) tb16k::tmem_dealloc<S::TM_COLS>(*tmem_slot);
    }
}

// std key polynomial (u64 torus, fft/mod.rs:197-218) -> the kernel's Fourier layout, scale 2^-64 / (N/2) folded in
template <int LOGN>
__global__ void __launch_bounds__(Shape<LOGN>::T)
bsk_convert_generic_kernel(const uint64_t *__restrict__ bsk_std, cplx *__restrict__ bskf, const cplx *__restrict__ tw) {
    using S = Shape<LOGN>;
    constexpr int N = S::N, M = S::M, PER = S::PER, T = S::T;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cplx *buf = reinterpret_cast<cplx *>(smem_raw);
    cplx *rt = buf + M;
    make_tables<M, T>(rt, tw, 2);
    const uint64_t *src = bsk_std + (size_t)blockIdx.x * N;
    const double scale = 1.0 / (18446744073709551616.0 * (double)M);
#pragma unroll
    for (int q = 0; q < PER; ++q) {
        const int j = threadIdx.x + T * q;
        cplx z;
        z.x = DMUL((double)(long long)src[j], scale);
        z.y = DMUL((double)(long long)src[j + M], scale);
        buf[SW(j)] = cmul(z, __ldg(tw + j));
    }
    fft_fwd<M, T>(buf, rt);
#pragma unroll
    for (int q = 0; q < PER; ++q) bskf[(size_t)blockIdx.x * M + threadIdx.x + T * q] = buf[SW(threadIdx.x + T * q)];
}

template <int LOGN, int K1, int GF>
cudaError_t launch(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskf, const void *tw,
                   uint64_t *out, const uint32_t *out_slot, tbk::ManyLut many, int batch, int n, int base_log, int levels, int n_iters, cudaStream_t stream) {
    using S = Shape<LOGN, K1>;
    using F = typename std::conditional<S::R8, Fft8<S::M, S::T>, Fft4<S::M, S::T>>::type;
    const size_t smem = (size_t)K1 * S::N * 8 + (size_t)S::M * 16 + (size_t)F::ENTRIES * 16 + 16;   // + the Tensor Memory base address slot
    // function attributes are per device: set on every launch (microseconds) rather than caching a process-wide flag
    cudaError_t e = cudaFuncSetAttribute(pbs_generic_kernel<LOGN, K1, GF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(pbs_generic_kernel<LOGN, K1, GF>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    pbs_generic_kernel<LOGN, K1, GF><<<batch, S::T, smem, stream>>>(lwe_small, lut_idx, luts, reinterpret_cast<const cplx *>(bskf),
                                                                 reinterpret_cast<const cplx *>(tw), out, out_slot, many, n, base_log, levels, n_iters);
    return cudaGetLastError();
}

template <int LOGN>
cudaError_t convert(const uint64_t *bsk_std, void *bskf, const void *tw, size_t n_polys, cudaStream_t stream) {
    using S = Shape<LOGN>;
    const size_t smem = (size_t)S::M * 16 + (size_t)Tables<S::M>::ENTRIES * 16;
    cudaError_t e = cudaFuncSetAttribute(bsk_convert_generic_kernel<LOGN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    bsk_convert_generic_kernel<LOGN><<<(unsigned)n_polys, S::T, smem, stream>>>(bsk_std, reinterpret_cast<cplx *>(bskf),
                                                                                 reinterpret_cast<const cplx *>(tw));
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------------------------
// N = 16384 and 32768 (PARAM_MESSAGE_1_CARRY_6 ... PARAM_MESSAGE_8_CARRY_0, mod.rs:913-1136): accumulator (up to 512 KiB), transform
// buffer and Fourier-domain outputs do not fit one SM's shared memory, so they live in a per-CTA global scratch area (L2 resident:
// 1.25 MiB per CTA) and only the FFT's inner stages run in shared memory: forward = log2(M / 4096) radix-2 stages through L2, then each
// contiguous 4096-point block is finished in a 64 KiB shared buffer; the inverse mirrors it.  Two 512-thread CTAs per SM, each walking
// over ciphertexts blockIdx.x, blockIdx.x + gridDim.x, ...
// ---------------------------------------------------------------------------------------------------------------------------------
constexpr int BIG_T = 512, BIG_CH = 4096;
using BigFft = Fft8<BIG_CH, BIG_T>;

// The last log2(4096) DIF stages of a size-M transform are complete 4096-point transforms of each contiguous block (the stage twiddle
// W_{2*half}^j does not depend on M), so the shared-memory part is fft_fwd / fft_inv of size BIG_CH with that size's root table.
template <int M>
__device__ __forceinline__ void fft_fwd_big(cplx *g, cplx *sm, const cplx *rt, const cplx *__restrict__ tw) {
    for (int half = M / 2; half >= BIG_CH; half >>= 1) {
        __syncthreads();
        const int stride = M / 2 / half;
        for (int b = threadIdx.x; b < M / 2; b += BIG_T) {
            const int j = b & (half - 1), i0 = ((b - j) << 1) + j, i1 = i0 + half;
            const cplx u = g[i0], v = g[i1];
            g[i0] = cadd(u, v);
            g[i1] = cmul(csub(u, v), root<M>(tw, j * stride));
        }
    }
    for (int c0 = 0; c0 < M; c0 += BIG_CH) {
        __syncthreads();
        for (int j = threadIdx.x; j < BIG_CH; j += BIG_T) sm[BigFft::sw(j)] = g[c0 + j];
        BigFft::fwd(sm, rt);
        for (int j = threadIdx.x; j < BIG_CH; j += BIG_T) g[c0 + j] = sm[BigFft::sw(j)];
    }
    __syncthreads();
}

template <int M>
__device__ __forceinline__ void fft_inv_big(cplx *g, cplx *sm, const cplx *rt, const cplx *__restrict__ tw) {
    for (int c0 = 0; c0 < M; c0 += BIG_CH) {
        __syncthreads();
        for (int j = threadIdx.x; j < BIG_CH; j += BIG_T) sm[BigFft::sw(j)] = g[c0 + j];
        BigFft::inv(sm, rt);
        for (int j = threadIdx.x; j < BIG_CH; j += BIG_T) g[c0 + j] = sm[BigFft::sw(j)];
    }
    for (int half = BIG_CH; half <= M / 2; half <<= 1) {
        __syncthreads();
        const int stride = M / 2 / half;
        for (int b = threadIdx.x; b < M / 2; b += BIG_T) {
            const int j = b & (half - 1), i0 = ((b - j) << 1) + j, i1 = i0 + half;
            const cplx u = g[i0];
            const cplx v = cmul_conj(g[i1], root<M>(tw, j * stride));
            g[i0] = cadd(u, v);
            g[i1] = csub(u, v);
        }
    }
    __syncthreads();
}

template <int LOGN, int K1>
__host__ __device__ constexpr size_t big_scratch_bytes() { return (size_t)K1 * (1 << LOGN) * 8 + (size_t)(1 << (LOGN - 1)) * 16 * (1 + K1); }

template <int LOGN, int K1>
__global__ void __launch_bounds__(BIG_T, 2)
pbs_generic_big_kernel(const uint64_t *__restrict__ lwe_small, const uint32_t *__restrict__ lut_idx, const uint64_t *__restrict__ luts,
                       const cplx *__restrict__ bskf, const cplx *__restrict__ tw, uint64_t *__restrict__ out,
                       const uint32_t *__restrict__ out_slot, const tbk::ManyLut many, unsigned char *scratch, int batch, int n, int base_log, int levels,
                       int n_iters) {
    constexpr int N = 1 << LOGN, M = N / 2, T = BIG_T;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cplx *sm = reinterpret_cast<cplx *>(smem_raw);                                              // [BIG_CH]
    cplx *rt = sm + BIG_CH;                                                                     // [BigFft::ENTRIES]
    BigFft::make(rt, tw, N / BIG_CH);
    unsigned char *mine = scratch + (size_t)blockIdx.x * big_scratch_bytes<LOGN, K1>();
    uint64_t *acc = reinterpret_cast<uint64_t *>(mine);                                         // [K1][N]
    cplx *buf = reinterpret_cast<cplx *>(mine + (size_t)K1 * N * 8);                            // [M]
    cplx *o = buf + M;                                                                          // [K1][M]
    const int t = threadIdx.x;
    const auto mod_switch = [](uint64_t x) { return (uint32_t)(((x >> (64 - LOGN - 2)) + 1) >> 1) & (2 * N - 1); };

    for (int ct = blockIdx.x; ct < batch; ct += gridDim.x) {
        const uint64_t *lwe = lwe_small + (size_t)ct * (n + 1);
        {
            const uint32_t a0 = (2 * N - mod_switch(__ldg(lwe + n))) & (2 * N - 1);
            const uint64_t *lut = luts + (size_t)(lut_idx ? lut_idx[ct] : 0) * K1 * N;
            for (int c = 0; c < K1; ++c)
                for (int j = t; j < N; j += T) {
                    const uint32_t s = ((uint32_t)j - a0) & (2 * N - 1);
                    const uint64_t v = __ldg(lut + c * N + (s & (N - 1)));
                    acc[c * N + j] = s >= (uint32_t)N ? (uint64_t)0 - v : v;
                }
        }
        __syncthreads();
        for (int i = 0; i < n_iters; ++i) {
            const uint32_t a_hat = mod_switch(__ldg(lwe + i));
            if (a_hat == 0) continue;
            for (int e = t; e < K1 * M; e += T) { o[e].x = 0.0; o[e].y = 0.0; }
            const cplx *ggsw = bskf + (size_t)i * levels * K1 * K1 * M;
            for (int lv = levels; lv >= 1; --lv) {
                for (int r = 0; r < K1; ++r) {
                    const uint64_t *src = acc + r * N;
                    for (int j = t; j < M; j += T) {
                        const uint32_t s0 = ((uint32_t)j - a_hat) & (2 * N - 1), s1 = ((uint32_t)(j + M) - a_hat) & (2 * N - 1);
                        uint64_t v0 = src[s0 & (N - 1)], v1 = src[s1 & (N - 1)];
                        v0 = (s0 >= (uint32_t)N ? (uint64_t)0 - v0 : v0) - src[j];
                        v1 = (s1 >= (uint32_t)N ? (uint64_t)0 - v1 : v1) - src[j + M];
                        cplx z;
                        z.x = (double)signed_digit(v0, base_log, levels, lv);
                        z.y = (double)signed_digit(v1, base_log, levels, lv);
                        buf[j] = cmul(z, __ldg(tw + j));
                    }
                    fft_fwd_big<M>(buf, sm, rt, tw);
                    const cplx *g = ggsw + ((size_t)(lv - 1) * K1 + r) * K1 * M;
                    for (int pos = t; pos < M; pos += T) {
                        const cplx f = buf[pos];
#pragma unroll
                        for (int c = 0; c < K1; ++c) {
                            const cplx gv = __ldg(g + (size_t)c * M + pos);
                            cplx a = o[c * M + pos];
                            a.x = DFMA(f.x, gv.x, DFMA(-f.y, gv.y, a.x));
                            a.y = DFMA(f.x, gv.y, DFMA(f.y, gv.x, a.y));
                            o[c * M + pos] = a;
                        }
                    }
                    __syncthreads();
                }
            }
            for (int c = 0; c < K1; ++c) {
                fft_inv_big<M>(o + c * M, sm, rt, tw);
                for (int j = t; j < M; j += T) {
                    const cplx z = cmul_conj(o[c * M + j], __ldg(tw + j));
                    acc[c * N + j] += tb::from_torus_f64(z.x);
                    acc[c * N + j + M] += tb::from_torus_f64(z.y);
                }
            }
            __syncthreads();
        }
        if (many.fn) {
            const int nf = tbx::many_fn_count(many, lut_idx, ct);
            tbx::extract_many_acc(out, out_slot[ct], nf, tbx::many_step(many, nf, N), acc, N, K1 - 1, t, T);
        } else {
            uint64_t *dst = out + (size_t)(out_slot ? out_slot[ct] : ct) * ((size_t)(K1 - 1) * N + 1);
            for (int r = 0; r < K1 - 1; ++r)
                for (int j = t; j < N; j += T) dst[r * N + j] = j == 0 ? acc[r * N] : (uint64_t)0 - acc[r * N + N - j];
            if (t == 0) dst[(K1 - 1) * N] = acc[(K1 - 1) * N];
        }
        __syncthreads();      // the next ciphertext overwrites the accumulator
    }
}

template <int LOGN>
__global__ void __launch_bounds__(BIG_T)
bsk_convert_generic_big_kernel(const uint64_t *__restrict__ bsk_std, cplx *bskf, const cplx *__restrict__ tw) {
    constexpr int N = 1 << LOGN, M = N / 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cplx *sm = reinterpret_cast<cplx *>(smem_raw);
    cplx *rt = sm + BIG_CH;
    BigFft::make(rt, tw, N / BIG_CH);
    const uint64_t *src = bsk_std + (size_t)blockIdx.x * N;
    cplx *dst = bskf + (size_t)blockIdx.x * M;            // transformed in place
    const double scale = 1.0 / (18446744073709551616.0 * (double)M);
    for (int j = threadIdx.x; j < M; j += BIG_T) {
        cplx z;
        z.x = DMUL((double)(long long)src[j], scale);
        z.y = DMUL((double)(long long)src[j + M], scale);
        dst[j] = cmul(z, __ldg(tw + j));
    }
    fft_fwd_big<M>(dst, sm, rt, tw);
}

template <int LOGN, int K1>
cudaError_t launch_big(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskf, const void *tw,
                       uint64_t *out, const uint32_t *out_slot, tbk::ManyLut many, int batch, int n, int base_log, int levels, int n_iters, cudaStream_t stream) {
    const size_t smem = (size_t)BIG_CH * 16 + (size_t)BigFft::ENTRIES * 16;
    cudaError_t e = cudaFuncSetAttribute(pbs_generic_big_kernel<LOGN, K1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int dev = 0, sms = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    const int grid = batch < 2 * sms ? batch : 2 * sms;
    unsigned char *scratch = nullptr;     // stream-ordered: concurrent launches on other streams get their own area
    if ((e = cudaMallocAsync((void **)&scratch, (size_t)grid * big_scratch_bytes<LOGN, K1>(), stream)) != cudaSuccess) return e;
    pbs_generic_big_kernel<LOGN, K1><<<grid, BIG_T, smem, stream>>>(lwe_small, lut_idx, luts, reinterpret_cast<const cplx *>(bskf),
                                                                    reinterpret_cast<const cplx *>(tw), out, out_slot, many, scratch, batch, n,
                                                                    base_log, levels, n_iters);
    e = cudaGetLastError();
    const cudaError_t e2 = cudaFreeAsync(scratch, stream);
    return e != cudaSuccess ? e : e2;
}

template <int LOGN>
cudaError_t convert_big(const uint64_t *bsk_std, void *bskf, const void *tw, size_t n_polys, cudaStream_t stream) {
    const size_t smem = (size_t)BIG_CH * 16 + (size_t)BigFft::ENTRIES * 16;
    cudaError_t e = cudaFuncSetAttribute(bsk_convert_generic_big_kernel<LOGN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    bsk_convert_generic_big_kernel<LOGN><<<(unsigned)n_polys, BIG_T, smem, stream>>>(bsk_std, reinterpret_cast<cplx *>(bskf),
                                                                                     reinterpret_cast<const cplx *>(tw));
    return cudaGetLastError();
}

}  // namespace tbg

namespace tbk {

// (polynomial size, GLWE dimension) pairs of shortint/parameters/mod.rs with N <= 8192
#define TBG_SHAPES(X) X(8, 5) X(9, 3) X(9, 2) X(10, 2) X(11, 1) X(12, 1) X(13, 1)

bool pbs_generic_supported(int poly_size, int glwe_dim) {
#define X(LOGN, K) if (poly_size == (1 << LOGN) && glwe_dim == K) return true;
    TBG_SHAPES(X)
#undef X
    return glwe_dim == 1 && (poly_size == 16384 || poly_size == 32768);
}

cudaError_t launch_pbs_generic(const uint64_t *lwe_small, const uint32_t *lut_idx, const uint64_t *luts, const void *bskf, const void *tw,
                               uint64_t *out, const uint32_t *out_slot, tbk::ManyLut many, int batch, int n, int poly_size, int glwe_dim, int base_log,
                               int levels, int grouping_factor, int n_iters, cudaStream_t stream) {
    if (batch <= 0) return cudaSuccess;
#define X(LOGN, K)                                                                                                                   \
    if (poly_size == (1 << LOGN) && glwe_dim == K) {                                                                                 \
        if (grouping_factor == 0)                                                                                                    \
            return tbg::launch<LOGN, K + 1, 0>(lwe_small, lut_idx, luts, bskf, tw, out, out_slot, many, batch, n, base_log, levels, n_iters, stream); \
        if (grouping_factor == 2)                                                                                                    \
            return tbg::launch<LOGN, K + 1, 2>(lwe_small, lut_idx, luts, bskf, tw, out, out_slot, many, batch, n, base_log, levels, n_iters, stream); \
        if (grouping_factor == 3)                                                                                                    \
            return tbg::launch<LOGN, K + 1, 3>(lwe_small, lut_idx, luts, bskf, tw, out, out_slot, many, batch, n, base_log, levels, n_iters, stream); \
        return cudaErrorInvalidValue;                                                                                                \
    }
    TBG_SHAPES(X)
#undef X
    if (grouping_factor != 0) return cudaErrorInvalidValue;
    if (glwe_dim == 1 && poly_size == 16384)
        return tbg::launch_big<14, 2>(lwe_small, lut_idx, luts, bskf, tw, out, out_slot, many, batch, n, base_log, levels, n_iters, stream);
    if (glwe_dim == 1 && poly_size == 32768)
        return tbg::launch_big<15, 2>(lwe_small, lut_idx, luts, bskf, tw, out, out_slot, many, batch, n, base_log, levels, n_iters, stream);
    return cudaErrorInvalidValue;
}

cudaError_t launch_bsk_convert_generic(const uint64_t *bsk_std, void *bskf, const void *tw, size_t n_polys, int poly_size, cudaStream_t stream) {
    switch (poly_size) {
    case 256: return tbg::convert<8>(bsk_std, bskf, tw, n_polys, stream);
    case 512: return tbg::convert<9>(bsk_std, bskf, tw, n_polys, stream);
    case 1024: return tbg::convert<10>(bsk_std, bskf, tw, n_polys, stream);
    case 2048: return tbg::convert<11>(bsk_std, bskf, tw, n_polys, stream);
    case 4096: return tbg::convert<12>(bsk_std, bskf, tw, n_polys, stream);
    case 8192: return tbg::convert<13>(bsk_std, bskf, tw, n_polys, stream);
    case 16384: return tbg::convert_big<14>(bsk_std, bskf, tw, n_polys, stream);
    case 32768: return tbg::convert_big<15>(bsk_std, bskf, tw, n_polys, stream);
    }
    return cudaErrorInvalidValue;
}

}  // namespace tbk
