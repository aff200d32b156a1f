// fft_core.cuh -- per-thread pieces of the size-1024 complex FFT that carries the negacyclic
// product of degree-2048 torus polynomials (the transform behind tfhe-rs
// core_crypto/fft_impl/fft64/math/fft/mod.rs:220-326,496-557, i.e. concrete-fft's plan.fwd/plan.inv
// plus the fold/twist conversions).
//
// Layout (B200-first, not concrete-fft's): one WARP owns one polynomial; lane l holds the 32 complex
// points j = l + 32*m (m = register index), i.e. 64 FP64 registers per thread.  The transform is a
// 32 x 32 four-step:
//   pass 1  in-register radix-2 DIF over m of z_j * w^(32 m)   (w = exp(i*pi/2048): the negacyclic twist,
//           its m-dependent part is a compile-time constant)
//   twiddle register p, lane l  *=  T[p][l] = w^l * W^(l * brev5(p))          (W = exp(-2*pi*i/1024))
//   one transpose through a warp-private shared-memory tile (lane <-> register)
//   pass 2  in-register radix-2 DIF
// so thread t, register p ends up holding frequency k = brev5(t) + 32*brev5(p).  The inverse runs the
// same steps backwards with conjugated twiddles (DIT), so no reordering is ever needed: the Fourier
// bootstrapping key is produced by this very code and is multiplied point-wise in the same layout.
//
// The file compiles both under nvcc (device code) and a plain C++ compiler (tests/cpu_mirror builds a
// lane-by-lane emulation from it to check the index algebra without a GPU).  All FP64 operations go
// through D* macros that map to non-contracting intrinsics on the device and to plain IEEE operations
// on the host (compile the host side with -ffp-contract=off), so both produce identical bits.
#pragma once
#include <cmath>
#include <cstdint>

#if defined(__CUDACC__)
#define TB_HD __host__ __device__ __forceinline__
#else
#define TB_HD inline
#endif

#if defined(__CUDA_ARCH__)
#define DMUL(a, b) __dmul_rn((a), (b))
#define DADD(a, b) __dadd_rn((a), (b))
#define DSUB(a, b) __dadd_rn((a), -(b))
#define DFMA(a, b, c) __fma_rn((a), (b), (c))
#else
#define DMUL(a, b) ((a) * (b))
#define DADD(a, b) ((a) + (b))
#define DSUB(a, b) ((a) - (b))
#define DFMA(a, b, c) std::fma((a), (b), (c))
#endif

namespace tb {

#if defined(__CUDACC__)
using cplx = double2;
#else
struct alignas(16) cplx { double x, y; };
#endif

constexpr int kLogN = 11;
constexpr int kN = 1 << kLogN;      // polynomial size handled by this FFT
constexpr int kM = kN / 2;          // complex points
constexpr int kR = 32;              // points per thread == lanes per polynomial

TB_HD constexpr int brev5(int x) {
    return ((x & 1) << 4) | ((x & 2) << 2) | (x & 4) | ((x & 8) >> 2) | ((x & 16) >> 4);
}

// cos(2*pi*j/32), sin(2*pi*j/32) for j = 0..15
TB_HD constexpr double w32_cos(int j) {
    constexpr double t[16] = {1.0,
                              0.98078528040323044913, 0.92387953251128675613, 0.83146961230254523708,
                              0.7071067811865475244, 0.55557023301960222474, 0.38268343236508977173,
                              0.19509032201612826785, 0.0,
                              -0.19509032201612826785, -0.38268343236508977173, -0.55557023301960222474,
                              -0.7071067811865475244, -0.83146961230254523708, -0.92387953251128675613,
                              -0.98078528040323044913};
    return t[j];
}
TB_HD constexpr double w32_sin(int j) {
    constexpr double t[16] = {0.0,
                              0.19509032201612826785, 0.38268343236508977173, 0.55557023301960222474,
                              0.7071067811865475244, 0.83146961230254523708, 0.92387953251128675613,
                              0.98078528040323044913, 1.0,
                              0.98078528040323044913, 0.92387953251128675613, 0.83146961230254523708,
                              0.7071067811865475244, 0.55557023301960222474, 0.38268343236508977173,
                              0.19509032201612826785};
    return t[j];
}
// negacyclic pre-twist w^(32 m) = exp(i*pi*m/64), m = 0..31
TB_HD constexpr double pre_cos(int m) {
    constexpr double t[32] = {1.0, 0.99879545620517239271, 0.99518472667219688624, 0.98917650996478097345,
                              0.98078528040323044913, 0.9700312531945439926, 0.95694033573220886494,
                              0.94154406518302077841, 0.92387953251128675613, 0.90398929312344333159,
                              0.88192126434835502971, 0.8577286100002720699, 0.83146961230254523708,
                              0.80320753148064490981, 0.77301045336273696081, 0.74095112535495909118,
                              0.7071067811865475244, 0.67155895484701840063, 0.63439328416364549822,
                              0.59569930449243334347, 0.55557023301960222474, 0.51410274419322172659,
                              0.47139673682599764856, 0.42755509343028209432, 0.38268343236508977173,
                              0.33688985339222005069, 0.29028467725446236764, 0.24298017990326388995,
                              0.19509032201612826785, 0.14673047445536175166, 0.098017140329560601994,
                              0.049067674327418014255};
    return t[m];
}
TB_HD constexpr double pre_sin(int m) { return m == 0 ? 0.0 : pre_cos(32 - m == 32 ? 0 : 32 - m); }

// ---- in-register 32-point DFT, radix-2 DIF, natural in -> bit-reversed out (kernel exp(-2*pi*i*m*q/32)) ----
template <int H>
TB_HD void dif_stage(double (&re)[32], double (&im)[32]) {
#pragma unroll
    for (int b = 0; b < 32; b += 2 * H) {
#pragma unroll
        for (int j = 0; j < H; ++j) {
            const int i0 = b + j, i1 = b + j + H;
            const int e = j * (16 / H);  // W_{2H}^j = W32^e
            const double ur = re[i0], ui = im[i0], vr = re[i1], vi = im[i1];
            re[i0] = DADD(ur, vr);
            im[i0] = DADD(ui, vi);
            const double dr = DSUB(ur, vr), di = DSUB(ui, vi);
            if (e == 0) {
                re[i1] = dr; im[i1] = di;
            } else if (e == 8) {          // times -i
                re[i1] = di; im[i1] = -dr;
            } else {                      // (dr + i di) * (c - i s)
                const double c = w32_cos(e), s = w32_sin(e);
                re[i1] = DFMA(dr, c, DMUL(di, s));
                im[i1] = DFMA(di, c, -DMUL(dr, s));
            }
        }
    }
}

TB_HD void radix32_dif(double (&re)[32], double (&im)[32]) {
    dif_stage<16>(re, im);
    dif_stage<8>(re, im);
    dif_stage<4>(re, im);
    dif_stage<2>(re, im);
    dif_stage<1>(re, im);
}

// ---- exact inverse of radix32_dif up to a factor 32: radix-2 DIT, bit-reversed in -> natural out ----
template <int H>
TB_HD void dit_stage_inv(double (&re)[32], double (&im)[32]) {
#pragma unroll
    for (int b = 0; b < 32; b += 2 * H) {
#pragma unroll
        for (int j = 0; j < H; ++j) {
            const int i0 = b + j, i1 = b + j + H;
            const int e = j * (16 / H);
            const double ur = re[i0], ui = im[i0], xr = re[i1], xi = im[i1];
            if (e == 0 || e == 8) {
                double vr, vi;
                if (e == 0) { vr = xr; vi = xi; } else { vr = -xi; vi = xr; }   // times 1 / times +i
                re[i0] = DADD(ur, vr);
                im[i0] = DADD(ui, vi);
                re[i1] = DSUB(ur, vr);
                im[i1] = DSUB(ui, vi);
            } else {
                // u +- x * (c + i s) with the cosine factored out (t = s / c): 6 FMAs instead of 2 mul + 2 fma + 4 add
                const double c = w32_cos(e), t = w32_sin(e) / w32_cos(e);
                const double p = DFMA(-t, xi, xr);      // (x * (1 + i t)).re
                const double q = DFMA(t, xr, xi);       // (x * (1 + i t)).im
                re[i0] = DFMA(c, p, ur);
                im[i0] = DFMA(c, q, ui);
                re[i1] = DFMA(-c, p, ur);
                im[i1] = DFMA(-c, q, ui);
            }
        }
    }
}

TB_HD void radix32_dit_inv(double (&re)[32], double (&im)[32]) {
    dit_stage_inv<1>(re, im);
    dit_stage_inv<2>(re, im);
    dit_stage_inv<4>(re, im);
    dit_stage_inv<8>(re, im);
    dit_stage_inv<16>(re, im);
}

// z[m] *= exp(+i*pi*m/64)   (forward negacyclic twist, register-dependent part)
TB_HD void pretwist_fwd(double (&re)[32], double (&im)[32]) {
#pragma unroll
    for (int m = 1; m < 32; ++m) {
        const double c = pre_cos(m), s = pre_sin(m);
        const double a = re[m], b = im[m];
        if (m == 16) {   // (a + ib)(1 + i)/sqrt2
            re[m] = DMUL(DSUB(a, b), c);
            im[m] = DMUL(DADD(a, b), c);
        } else {
            re[m] = DFMA(a, c, -DMUL(b, s));
            im[m] = DFMA(b, c, DMUL(a, s));
        }
    }
}

// z[m] *= exp(-i*pi*m/64)   (inverse)
TB_HD void posttwist_inv(double (&re)[32], double (&im)[32]) {
#pragma unroll
    for (int m = 1; m < 32; ++m) {
        const double c = pre_cos(m), s = pre_sin(m);
        const double a = re[m], b = im[m];
        if (m == 16) {   // (a + ib)(1 - i)/sqrt2
            re[m] = DMUL(DADD(a, b), c);
            im[m] = DMUL(DSUB(b, a), c);
        } else {
            re[m] = DFMA(a, c, DMUL(b, s));
            im[m] = DFMA(b, c, -DMUL(a, s));
        }
    }
}

// The inter-pass twiddle table: tbl[p*32 + l] = w^l * W^(l*brev5(p)) = exp(i*pi*l*(1 - 4*brev5(p))/2048),
// stored as interleaved (re, im).  Built on the host in long double (see tb_make_twiddle_table).
// register p of lane l *= tbl[p*32 + l]   (forward)   /   *= conj(tbl[p*32 + l])   (inverse)
// Loads are issued in groups of TB_TW_CHUNK so that the compiler cannot hoist all 32 (128 registers)
// above the butterflies and spill; TB_FENCE stops it from merging the groups.
#if defined(__CUDA_ARCH__)
#define TB_FENCE() asm volatile("" ::: "memory")
#else
#define TB_FENCE() do {} while (0)
#endif
constexpr int TB_TW_CHUNK = 8;

template <class Load>
TB_HD void twiddle_fwd(double (&re)[32], double (&im)[32], Load load, int lane) {
#pragma unroll
    for (int c = 0; c < 32; c += TB_TW_CHUNK) {
        cplx w[TB_TW_CHUNK];
#pragma unroll
        for (int q = 0; q < TB_TW_CHUNK; ++q) w[q] = load((c + q) * 32 + lane);
#pragma unroll
        for (int q = 0; q < TB_TW_CHUNK; ++q) {
            const double a = re[c + q], b = im[c + q];
            re[c + q] = DFMA(a, w[q].x, -DMUL(b, w[q].y));
            im[c + q] = DFMA(b, w[q].x, DMUL(a, w[q].y));
        }
        TB_FENCE();
    }
}
template <class Load>
TB_HD void twiddle_inv(double (&re)[32], double (&im)[32], Load load, int lane) {
#pragma unroll
    for (int c = 0; c < 32; c += TB_TW_CHUNK) {
        cplx w[TB_TW_CHUNK];
#pragma unroll
        for (int q = 0; q < TB_TW_CHUNK; ++q) w[q] = load((c + q) * 32 + lane);
#pragma unroll
        for (int q = 0; q < TB_TW_CHUNK; ++q) {
            const double a = re[c + q], b = im[c + q];
            re[c + q] = DFMA(a, w[q].x, DMUL(b, w[q].y));
            im[c + q] = DFMA(b, w[q].x, -DMUL(a, w[q].y));
        }
        TB_FENCE();
    }
}

// shared-memory transpose addressing: a 32 x 33 (padded) tile of 8-byte words.  (lane L, register r) is
// written at word r*33 + L; afterwards lane L reads register r from word L*33 + r.  Every address is
// "per-lane base + compile-time constant" (no per-register index registers to keep alive across the
// blind-rotation loop) and both sides are bank-conflict free (33 = 1 mod 16 for 8-byte words).
constexpr int kXposeStride = 33;
constexpr int kXposeWords = 32 * kXposeStride;
TB_HD constexpr int xpose_write_idx(int lane, int r) { return r * kXposeStride + lane; }
TB_HD constexpr int xpose_read_idx(int lane, int r) { return lane * kXposeStride + r; }

// frequency held by (thread t, register p) after the forward transform
TB_HD constexpr int freq_of(int t, int p) { return brev5(t) + 32 * brev5(p); }

// ---- integer helpers of the blind rotation -------------------------------------------------------

// fft_impl/common.rs:26-43 fast_pbs_modulus_switch for N = 2048 (value in [0, 2N])
TB_HD uint32_t modulus_switch_2n(uint64_t x) { return (uint32_t)(((x >> (64 - kLogN - 2)) + 1) >> 1); }

// signed digit of the 1-level decomposition (decomposer.rs:98-118 then iter.rs:120-127 with level = 1):
// round x to its top base_log bits; the representative lies in (-B/2, B/2].
TB_HD int32_t signed_digit_l1(uint64_t x, int base_log) {
    const uint32_t hi = (uint32_t)(x >> 32);
    const uint32_t t = hi >> (31 - base_log);
    const uint32_t r = ((t + 1u) >> 1) & ((1u << base_log) - 1u);
    const uint32_t half = 1u << (base_log - 1);
    return (int32_t)r - (int32_t)((r > half) ? (1u << base_log) : 0u);
}

// Gather of the rotated polynomial: u = (j - a) << (31 - kLogN) carries the source index d = (j - a) mod 2N with its wrap bit
// (d >= N: the word enters negated) on top.  Returns poly[d mod N] and sets `wrap` to all ones for a wrapped word, else 0; both are
// shifts of u (no index masking, no 64-bit negation), and u for j + c is u + (c << (31 - kLogN)).
TB_HD uint64_t rot_gather(const uint64_t *poly, uint32_t u, uint32_t &wrap) {
    wrap = (uint32_t)((int32_t)u >> 31);
    return *reinterpret_cast<const uint64_t *>(reinterpret_cast<const char *>(poly) + ((u << 1) >> (29 - kLogN)));
}

// signed_digit_l1(+-r - o, base_log) of the rotated gather (r: gathered word, wrap: rot_gather's mask, all ones when r enters
// negated; o: own word),
// computed from the high word of the complement only:
//   ~(+-r - o) = o + (r ^ ~M) + M,  M = wrap in both words          (one three-input add with carry)
//   signed_digit_l1(x) = -( (int32)(hi(~x) + 2^(31-B)) >> (32-B) )  (rounding half up on x is rounding half down on -x, and the
//                                                                    arithmetic shift lands in [-B/2, B/2): no tie fix-up)
// For 2 <= base_log <= 30 it equals signed_digit_l1 for every input (tests/test_rot_digit.py checks the classes that matter).
TB_HD int32_t rot_sub_digit(uint64_t r, uint32_t wrap, uint64_t o, int base_log) {
    uint32_t xl = (uint32_t)r, xh = (uint32_t)(r >> 32);
#if defined(__CUDA_ARCH__)
    // one LOP3 per word (the compiler splits ~(a ^ b) into two)
    asm("lop3.b32 %0, %0, %2, 0, 0xC3;\n\tlop3.b32 %1, %1, %2, 0, 0xC3;" : "+r"(xl), "+r"(xh) : "r"(wrap));
#else
    xl = ~(xl ^ wrap); xh = ~(xh ^ wrap);
#endif
    const uint64_t M = ((uint64_t)wrap << 32) | wrap;
    const uint32_t nh = (uint32_t)((o + (((uint64_t)xh << 32) | xl) + M) >> 32);
    return -((int32_t)(nh + (1u << (31 - base_log))) >> (32 - base_log));
}

// commons/math/torus/mod.rs:72-78 with the x86 rounding the reference actually runs (half-to-even,
// fft/x86.rs:859-867): fract = t - rint(t); (i64) rint(fract * 2^64).
TB_HD uint64_t from_torus_f64(double t) {
#if defined(__CUDA_ARCH__)
    const double fr = __dadd_rn(t, -rint(t));
    return (uint64_t)__double2ll_rn(__dmul_rn(fr, 18446744073709551616.0));
#else
    const double fr = t - std::nearbyint(t);
    const double sc = std::nearbyint(fr * 18446744073709551616.0);
    // |sc| <= 2^63; +2^63 (fract exactly 0.5) saturates like `as i64` and __double2ll_rn
    return sc >= 9223372036854775808.0 ? 0x7FFFFFFFFFFFFFFFULL : (uint64_t)(int64_t)sc;
#endif
}

// Coefficient j of (poly * X^a) for a in [0, 2N): +-poly[(j - a) mod N] (polynomial_algorithms.rs:219-270).
// Returns the source index and whether the value is negated.
TB_HD void rot_src(int j, uint32_t a, int &src, bool &neg) {
    const uint32_t s = ((uint32_t)j - a) & (2 * kN - 1);
    src = (int)(s & (kN - 1));
    neg = s >= (uint32_t)kN;
}

}  // namespace tb

// host-side builder of the inter-pass twiddle table (1024 double2)
static inline void tb_make_twiddle_table(double *interleaved /* 2*1024 */) {
    const long double pi = 3.14159265358979323846264338327950288L;
    for (int p = 0; p < 32; ++p)
        for (int l = 0; l < 32; ++l) {
            // exponent l*(1 - 4*k1) over 2048, reduced mod 4096 to keep the argument small
            long e = ((long)l * (1 - 4 * (long)tb::brev5(p))) % 4096;
            if (e < 0) e += 4096;
            const long double ang = pi * (long double)e / 2048.0L;
            interleaved[2 * (p * 32 + l)] = (double)cosl(ang);
            interleaved[2 * (p * 32 + l) + 1] = (double)sinl(ang);
        }
}
