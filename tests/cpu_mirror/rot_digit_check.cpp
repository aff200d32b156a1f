// The rotated-gather digit of the wide blind-rotation kernels (fft_core.cuh: rot_gather + rot_sub_digit) against the
// definition they replace: signed_digit_l1(+-poly[d mod N] - o, base_log), negated when d mod 2N >= N.
//   - rot_gather: every source index d mod 2N, and the index algebra u(j + c) = u(j) + (c << (31 - kLogN)) of the kernels' loops
//   - rot_sub_digit, for every base_log 2..30 the engine accepts:
//       ties at +-B/2 and the digits B/2 +- 1 around them, with the low-order remainder at -1, 0, +1 of the half step;
//       the words 0, 1, 2^63, 2^64 - 1 for the gathered and the own word;
//       borrow and no borrow from the low word (own words whose low half lies below / above the gathered word's);
//       both wrap flags;
//     then 10^7 random (gathered, own, wrap, base_log) tuples.
// Built with -DWRONG_TIE, the function under test keeps the tie at -B/2 instead of +B/2; the checker must then fail.
#include "../../fhe_string_bounty_b200/csrc/fft_core.cuh"
#include <cstdio>
#include <cstdlib>
#include <vector>

using namespace tb;

static int32_t digit_under_test(uint64_t r, uint32_t wrap, uint64_t o, int B) {
#ifdef WRONG_TIE
    const uint64_t x = (wrap ? (uint64_t)0 - r : r) - o;
    return (int32_t)((uint32_t)(x >> 32) + (1u << (31 - B))) >> (32 - B);   // representative in [-B/2, B/2)
#else
    return rot_sub_digit(r, wrap, o, B);
#endif
}

static int32_t reference(uint64_t r, bool neg, uint64_t o, int B) { return signed_digit_l1((neg ? (uint64_t)0 - r : r) - o, B); }

static long long checked = 0, failed = 0;

static void check(uint64_t r, bool neg, uint64_t o, int B) {
    ++checked;
    const int32_t want = reference(r, neg, o, B), got = digit_under_test(r, neg ? ~0u : 0u, o, B);
    if (got != want && failed++ < 10)
        std::printf("mismatch: r=%016llx neg=%d o=%016llx B=%d: got %d want %d\n", (unsigned long long)r, (int)neg,
                    (unsigned long long)o, B, got, want);
}

// the (r, neg) that makes +-r - o == x
static void check_x(uint64_t x, uint64_t o, int B) {
    const uint64_t s = x + o;
    check(s, false, o, B);
    check((uint64_t)0 - s, true, o, B);
}

static uint64_t splitmix(uint64_t &s) {
    uint64_t z = (s += 0x9E3779B97F4A7C15ULL);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

int main() {
    // rot_gather: poly[d mod N] and the wrap mask for every d mod 2N, from u = d << (31 - kLogN) built the way the kernels build it
    {
        std::vector<uint64_t> poly(kN);
        uint64_t s = 1;
        for (auto &v : poly) v = splitmix(s);
        for (uint32_t a = 0; a < 2 * kN; a += 7)
            for (int j = 0; j < kN / 2; ++j) {
                const uint32_t u = ((uint32_t)j - a) << (31 - kLogN);
                for (int c = 0; c < 2; ++c) {
                    const uint32_t d = ((uint32_t)(j + c * kM) - a) & (2 * kN - 1);
                    uint32_t wrap;
                    const uint64_t got = rot_gather(poly.data(), u + ((uint32_t)(c * kM) << (31 - kLogN)), wrap);
                    ++checked;
                    if (got != poly[d & (kN - 1)] || wrap != (d >= (uint32_t)kN ? ~0u : 0u)) {
                        if (failed++ < 10) std::printf("rot_gather mismatch: j=%d a=%u c=%d\n", j, a, c);
                    }
                }
            }
    }

    const uint64_t words[] = {0, 1, 1ULL << 63, ~0ULL, 0xFFFFFFFFULL, 1ULL << 32, (1ULL << 32) + 1, 0x7FFFFFFFFFFFFFFFULL,
                              0x8000000000000001ULL, 0xFFFFFFFF00000000ULL, 0x00000000FFFFFFFEULL, 0x123456789ABCDEF0ULL};
    for (int B = 2; B <= 30; ++B) {
        const uint64_t step = 1ULL << (64 - B), half = step >> 1, h = 1ULL << (B - 1), top = 1ULL << B;
        // digit classes: 0, +-1, +-(B/2 - 1), +-B/2 (the tie), B/2 + 1 (== -(B/2 - 1)), and the top digit
        const uint64_t cs[] = {0, 1, 2, h - 1, h, h + 1, top - h - 1, top - h, top - h + 1, top - 2, top - 1};
        // remainders below the digit: exact, one below / at / above the half step (ties), one below the next digit
        const uint64_t es[] = {0, 1, half - 1, half, half + 1, step - 1};
        for (uint64_t c : cs)
            for (uint64_t e : es) {
                const uint64_t x = c * step + e;
                for (uint64_t o : words) check_x(x, o, B);
                // borrow / no borrow: own word's low half just above / at / below the gathered word's low half
                for (uint64_t olo : {0ULL, 1ULL, 0x7FFFFFFFULL, 0x80000000ULL, 0xFFFFFFFEULL, 0xFFFFFFFFULL})
                    for (uint64_t ohi : {0ULL, 0x80000000ULL, 0xFFFFFFFFULL}) check_x(x, (ohi << 32) | olo, B);
            }
        for (uint64_t r : words)
            for (uint64_t o : words)
                for (int neg = 0; neg < 2; ++neg) check(r, neg, o, B);
    }

    uint64_t s = 0xB200;
    for (int i = 0; i < 10000000; ++i) {
        const uint64_t r = splitmix(s), o = splitmix(s), k = splitmix(s);
        check(r, k & 1, o, 2 + (int)((k >> 1) % 29));
    }

    if (failed) {
        std::printf("FAILED: %lld of %lld\n", failed, checked);
        return 1;
    }
    std::printf("OK: %lld cases\n", checked);
    return 0;
}
