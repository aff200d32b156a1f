// host/padded.h -- the part of the FheString surface whose RESULT LENGTH IS SECRET: strings in the null-padded model.
//
// A padded string has a public capacity and a secret length: the content is followed by zero bytes up to the capacity (once a zero
// byte appears every later byte is zero).  That is the model the bounty's FheString uses to hide lengths (SURVEY.md Appendix B, "API
// surface of the missing string module"); the reference snapshot itself only has the building blocks -- FheUint8 chars with
// to_upper / to_lower in docs/tutorials/ascii_fhe_string.md:81-154, and a zero-terminated-free Vec<RadixCiphertext> in
// examples/regex_engine/ciphertext.rs:4-22 / execution.rs:63-215 -- so, as for host/strings.h, only DECRYPTED results are comparable
// (against Rust's str semantics: len, is_empty, ==, <, trim_start / trim_end / trim with char::is_whitespace on ASCII, strip_prefix,
// strip_suffix, +, repeat, contains / starts_with / ends_with).
//
// Everything is composed from the radix methods of host/radix.h (count trees, comparator, cmux, carry-free one-hot sums) and recorded
// into the same level-batched programs: wide levels of independent KS-PBS jobs, which is what the engine is built for.  Secret shifts
// (trim_start, concat, strip_prefix with a padded pattern) are barrel shifters: one cmux level per bit of the shift amount
// (radix_parallel/cmux.rs:211-250), the amount itself being the radix index of a one-hot boundary flag, never a sum that could overflow
// a block.
#pragma once
#include <tuple>

#include "strings.h"

namespace tbh {

class PaddedStringServerKey {
  public:
    explicit PaddedStringServerKey(Program &prog) : pg(prog), isk(prog), ssk(prog), p(prog.params()) {
        ssk.require_two_bit_blocks("null-padded strings");
    }

    // ---- chars -----------------------------------------------------------------------------------------------------------------
    Radix trivial_char(unsigned char ch) {
        Radix c;
        for (size_t b = 0; b < 4; ++b) c.push_back(pg.create_trivial((ch >> (2 * b)) & 3));
        return c;
    }
    FheString extend(const FheString &s, size_t cap) {
        FheString r = s;
        while (r.len() < cap) r.chars.push_back(trivial_char(0));
        return r;
    }
    // b0 + b1 + b2 + b3 (<= 12): zero iff the char is the padding byte
    Ct block_sum(const Radix &c) {
        Ct s = c[0];
        for (size_t b = 1; b < c.size(); ++b) s = pg.unchecked_add(s, c[b]);
        return s;
    }
    BooleanBlock nonzero(const Radix &c) { return pg.pbs(block_sum(c), [](uint64_t x) { return uint64_t(x != 0); }); }
    BooleanBlock is_zero(const Radix &c) { return pg.pbs(block_sum(c), [](uint64_t x) { return uint64_t(x == 0); }); }
    // keep ? c : 0   (zero_out_if, radix_parallel/cmux.rs:281-)
    Radix keep_if(const Radix &c, const Ct &keep) {
        Radix r;
        for (auto &blk : c) r.push_back(pg.pbs_bivariate(blk, keep, [](uint64_t v, uint64_t k) { return (k & 1) ? v : uint64_t(0); }));
        return r;
    }
    // cond ? a : b per block (cmux.rs:211-250: two zero_out_if, add, message_extract)
    Radix select(const Ct &cond, const Radix &a, const Radix &b) { return isk.if_then_else(cond, a, b); }

    // ---- scans over boolean flags ---------------------------------------------------------------------------------------------
    // out[i] = OR_{j < i} f[j] (exclusive) or OR_{j <= i} f[j] (inclusive) in THREE levels: flags are cut into blocks of 14,
    //   level 1   any_k      = [sum of block k != 0]
    //   level 2   earlier_k  = [some block before k matched]     (running sums of <= 15 cleaned flags; a cleaned carry every group)
    //   level 3   out[i]     = [(flags of its block up to i) + earlier_k != 0]      (<= 14 + 1)
    std::vector<Ct> prefix_or(const std::vector<Ct> &f, bool inclusive) {
        const size_t n = f.size();
        std::vector<Ct> out(n);
        if (n == 0) return out;
        constexpr size_t BLK = 14;
        const size_t n_blk = (n + BLK - 1) / BLK, max_sum = p.total_mod() - 1;
        std::vector<Ct> any(n_blk), earlier(n_blk);
        for (size_t k = 0; k < n_blk; ++k) {
            Ct sum = f[k * BLK];
            for (size_t i = k * BLK + 1; i < std::min(n, (k + 1) * BLK); ++i) sum = pg.unchecked_add(sum, f[i]);
            any[k] = n_blk > 1 ? pg.pbs(sum, [](uint64_t x) { return uint64_t(x != 0); }) : sum;
        }
        earlier[0] = pg.create_trivial(0);
        Ct carry = pg.create_trivial(0);
        for (size_t g0 = 0; g0 < n_blk;) {
            const size_t g1 = std::min(n_blk, g0 + (g0 == 0 ? max_sum : max_sum - 1));
            Ct run = carry;
            for (size_t k = g0; k < g1; ++k) {
                if (k > 0) earlier[k] = pg.pbs(run, [](uint64_t x) { return uint64_t(x != 0); });
                run = pg.unchecked_add(run, any[k]);
            }
            if (g1 < n_blk) carry = pg.pbs(run, [](uint64_t x) { return uint64_t(x != 0); });
            g0 = g1;
        }
        for (size_t i = 0; i < n; ++i) {
            const size_t k = i / BLK;
            Ct y = earlier[k];
            for (size_t j = k * BLK; j < i + (inclusive ? 1 : 0); ++j) y = pg.unchecked_add(y, f[j]);
            out[i] = y.is_trivial() ? y : pg.pbs(y, [](uint64_t x) { return uint64_t(x != 0); });
        }
        return out;
    }
    // radix digits of the position of the single 1 in `onehot` (position w counts as value_of(w)); at most one flag is set, so the
    // selected digits are summed without carries, 15 at a time with a cleaning PBS (the chunking of scalar_comparison.rs:155-170)
    Radix onehot_to_radix(const std::vector<Ct> &onehot, size_t n_digits, const std::function<uint64_t(size_t)> &value_of) {
        const size_t max_value = p.total_mod() - 1;
        Radix digits;
        for (size_t d = 0; d < n_digits; ++d) {
            std::vector<Ct> terms;
            for (size_t w = 0; w < onehot.size(); ++w) {
                const uint64_t digit = (value_of(w) >> (2 * d)) & 3;
                if (digit == 0) continue;
                terms.push_back(pg.pbs(onehot[w], [digit](uint64_t x) { return (x & 1) ? digit : uint64_t(0); }));
            }
            if (terms.empty()) { digits.push_back(pg.create_trivial(0)); continue; }
            while (terms.size() > 1) {
                std::vector<Ct> next;
                for (size_t i = 0; i < terms.size(); i += max_value) {
                    const size_t len = std::min(max_value, terms.size() - i);
                    Ct sum = terms[i];
                    for (size_t j = 1; j < len; ++j) sum = pg.unchecked_add(sum, terms[i + j]);
                    sum.degree = p.msg_mod - 1;   // at most one term is non-zero
                    next.push_back(pg.pbs(sum, [this](uint64_t x) { return x % p.msg_mod; }));
                }
                terms.swap(next);
            }
            digits.push_back(terms[0]);
        }
        return digits;
    }
    static size_t digits_for(size_t max_value) {
        size_t d = 1;
        while ((size_t(1) << (2 * d)) <= max_value) ++d;
        return d;
    }
    // binary bits of a radix number, little-endian (2 per digit)
    std::vector<Ct> bits_of(const Radix &digits, size_t n_bits) {
        std::vector<Ct> bits;
        for (size_t d = 0; d < digits.size() && bits.size() < n_bits; ++d) {
            bits.push_back(pg.pbs(digits[d], [](uint64_t x) { return x & 1; }));
            if (bits.size() < n_bits) bits.push_back(pg.pbs(digits[d], [](uint64_t x) { return (x >> 1) & 1; }));
        }
        return bits;
    }
    // barrel shifter: s shifted by the secret amount sum_t bit_t 2^t (left: towards index 0, dropping chars; right: towards the end,
    // zero-filling), one cmux level per bit
    FheString shift(const FheString &s, const std::vector<Ct> &bits, bool left) {
        FheString cur = s;
        const size_t n = s.len();
        for (size_t t = 0; t < bits.size(); ++t) {
            const size_t k = size_t(1) << t;
            FheString nxt = cur;
            for (size_t i = 0; i < n; ++i) {
                const bool has_src = left ? (i + k < n) : (i >= k);
                if (has_src) nxt.chars[i] = select(bits[t], cur.chars[left ? i + k : i - k], cur.chars[i]);
                else nxt.chars[i] = keep_if(cur.chars[i], isk.boolean_bitnot(bits[t]));     // the shifted-in char is the padding byte
            }
            cur = nxt;
        }
        return cur;
    }

    // ---- len / is_empty ----------------------------------------------------------------------------------------------------------
    std::vector<Ct> nonzero_flags(const FheString &s) {
        std::vector<Ct> nz;
        for (auto &c : s.chars) nz.push_back(nonzero(c));
        return nz;
    }
    // boundary one-hot over positions 0 .. n: 1 at i == len
    std::vector<Ct> length_onehot(const std::vector<Ct> &nz) {
        const size_t n = nz.size();
        std::vector<Ct> b(n + 1);
        if (n == 0) { b[0] = pg.create_trivial(1); return b; }
        b[0] = isk.boolean_bitnot(nz[0]);
        for (size_t i = 1; i < n; ++i) {
            Ct y = pg.unchecked_add(nz[i - 1], pg.unchecked_scalar_mul(nz[i], 2));   // (prev, cur) = (1, 0) <=> y == 1
            b[i] = pg.pbs(y, [](uint64_t x) { return uint64_t(x == 1); });
        }
        b[n] = nz[n - 1];
        return b;
    }
    Radix len(const FheString &s) {
        return onehot_to_radix(length_onehot(nonzero_flags(s)), digits_for(s.len()), [](size_t w) { return uint64_t(w); });
    }
    BooleanBlock is_empty(const FheString &s) { return s.len() == 0 ? pg.create_trivial(1) : is_zero(s.chars[0]); }

    // ---- comparisons: the padding byte sorts below every char, so the unpadded circuits apply to the common capacity -------------------
    BooleanBlock eq(const FheString &a, const FheString &b) { const size_t n = std::max(a.len(), b.len()); return ssk.eq(extend(a, n), extend(b, n)); }
    BooleanBlock ne(const FheString &a, const FheString &b) { const size_t n = std::max(a.len(), b.len()); return ssk.ne(extend(a, n), extend(b, n)); }
    BooleanBlock lt(const FheString &a, const FheString &b) { const size_t n = std::max(a.len(), b.len()); return ssk.lt(extend(a, n), extend(b, n)); }
    BooleanBlock le(const FheString &a, const FheString &b) { const size_t n = std::max(a.len(), b.len()); return ssk.le(extend(a, n), extend(b, n)); }
    BooleanBlock gt(const FheString &a, const FheString &b) { const size_t n = std::max(a.len(), b.len()); return ssk.gt(extend(a, n), extend(b, n)); }
    BooleanBlock ge(const FheString &a, const FheString &b) { const size_t n = std::max(a.len(), b.len()); return ssk.ge(extend(a, n), extend(b, n)); }

    // ---- whitespace classes: 0 = other char, 1 = ASCII whitespace (U+0009 ..= U+000D, U+0020: char::is_whitespace), 2 = padding ------
    Ct char_class(const Radix &c) {
        Ct hi = pg.unchecked_add(pg.unchecked_scalar_mul(c[3], p.msg_mod), c[2]);
        Ct lo = pg.unchecked_add(pg.unchecked_scalar_mul(c[1], p.msg_mod), c[0]);
        Ct k = pg.pbs(hi, [](uint64_t x) { return x == 0 ? uint64_t(1) : (x == 2 ? uint64_t(2) : uint64_t(0)); });
        Ct r = pg.pbs(lo, [](uint64_t x) { return x == 0 ? uint64_t(2) : ((x >= 9 && x <= 13) ? uint64_t(1) : uint64_t(0)); });
        return pg.pbs_bivariate(k, r, [](uint64_t kk, uint64_t rr) {
            if (kk == 1 && rr == 2) return uint64_t(2);                        // 0x00
            if ((kk == 1 && rr == 1) || (kk == 2 && rr == 2)) return uint64_t(1);   // 0x09..0x0D, 0x20
            return uint64_t(0);
        });
    }
    FheString trim_end(const FheString &s) {
        const size_t n = s.len();
        if (n == 0) return s;
        std::vector<Ct> other(n);
        for (size_t i = 0; i < n; ++i) other[n - 1 - i] = pg.pbs(char_class(s.chars[i]), [](uint64_t x) { return uint64_t(x == 0); });
        std::vector<Ct> keep = prefix_or(other, true);      // over the reversed string: some non-whitespace char at or after i
        FheString out = s;
        for (size_t i = 0; i < n; ++i) out.chars[i] = keep_if(s.chars[i], keep[n - 1 - i]);
        return out;
    }
    FheString trim_start(const FheString &s) {
        const size_t n = s.len();
        if (n == 0) return s;
        std::vector<Ct> stop(n);                            // not whitespace: the first such char is where the result starts
        for (size_t i = 0; i < n; ++i) stop[i] = pg.pbs(char_class(s.chars[i]), [](uint64_t x) { return uint64_t(x != 1); });
        std::vector<Ct> before = prefix_or(stop, false);
        std::vector<Ct> first(n + 1);
        for (size_t i = 0; i < n; ++i) {
            Ct y = pg.unchecked_add(stop[i], pg.unchecked_scalar_mul(before[i], 2));
            first[i] = pg.pbs(y, [](uint64_t x) { return uint64_t(x == 1); });
        }
        {   // whitespace up to the capacity: everything goes
            Ct all = pg.unchecked_add(stop[n - 1], before[n - 1]);
            first[n] = pg.pbs(all, [](uint64_t x) { return uint64_t(x == 0); });
        }
        const size_t nd = digits_for(n);
        Radix amount = onehot_to_radix(first, nd, [](size_t w) { return uint64_t(w); });
        size_t n_bits = 1;
        while ((size_t(1) << n_bits) <= n) ++n_bits;
        return shift(s, bits_of(amount, n_bits), true);
    }
    FheString trim(const FheString &s) { return trim_end(trim_start(s)); }

    // ---- strip_prefix / strip_suffix with a clear pattern: (matched, string) -------------------------------------------------------------
    std::pair<BooleanBlock, FheString> strip_prefix(const FheString &s, const std::string &pat) {
        const size_t n = s.len(), m = pat.size();
        if (m == 0) return {pg.create_trivial(1), s};
        if (m > n) return {pg.create_trivial(0), s};
        BooleanBlock flag = ssk.starts_with(s, ssk.trivial_string(pat));
        FheString out = s;
        for (size_t i = 0; i < n; ++i)
            out.chars[i] = i + m < n ? select(flag, s.chars[i + m], s.chars[i]) : keep_if(s.chars[i], isk.boolean_bitnot(flag));
        return {flag, out};
    }
    // ends_with for a padded haystack: some window equals the pattern AND the string ends right after it
    BooleanBlock ends_with_clear(const FheString &s, const std::string &pat, const std::vector<Ct> &nz) {
        const size_t n = s.len(), m = pat.size();
        if (m == 0) return pg.create_trivial(1);
        if (m > n) return pg.create_trivial(0);
        FheString tp = ssk.trivial_string(pat);
        std::vector<Ct> per_window;
        for (size_t w = 0; w + m <= n; ++w) {
            std::vector<Ct> flags = isk.block_equalities(StringServerKey::concat(s, w, m), StringServerKey::concat(tp, 0, m));
            if (w + m < n) flags.push_back(isk.boolean_bitnot(nz[w + m]));
            per_window.push_back(isk.are_all_comparisons_block_true(flags));
        }
        return isk.is_at_least_one_comparisons_block_true(per_window);
    }
    std::pair<BooleanBlock, FheString> strip_suffix(const FheString &s, const std::string &pat) {
        const size_t n = s.len(), m = pat.size();
        if (m == 0) return {pg.create_trivial(1), s};
        if (m > n) return {pg.create_trivial(0), s};
        std::vector<Ct> nz = nonzero_flags(s);
        BooleanBlock flag = ends_with_clear(s, pat, nz);
        FheString out = s;
        for (size_t i = 0; i < n; ++i) {
            // char i belongs to the suffix iff the string ends within m chars of it: nz[i + m] == 0 (beyond the capacity: always)
            Ct keep = i + m < n ? pg.pbs_bivariate(flag, nz[i + m], [](uint64_t f, uint64_t z) { return uint64_t(!((f & 1) && !(z & 1))); })
                                : isk.boolean_bitnot(flag);
            out.chars[i] = keep_if(s.chars[i], keep);
        }
        return {flag, out};
    }

    // ---- pattern matching with a PADDED (secret-length) pattern ---------------------------------------------------------------------------
    // window w matches iff for every j: pat[j] is padding OR hay[w + j] == pat[j]  (chars beyond the haystack's capacity are padding)
    BooleanBlock window_match(const FheString &hay, const FheString &pat, size_t w, const std::vector<Ct> &pat_zero) {
        std::vector<Ct> ok;
        for (size_t j = 0; j < pat.len(); ++j) {
            if (w + j >= hay.len()) { ok.push_back(pat_zero[j]); continue; }
            std::vector<Ct> eqs = isk.block_equalities(hay.chars[w + j], pat.chars[j]);
            Ct y = pg.unchecked_scalar_mul(pat_zero[j], 4);
            for (auto &e : eqs) y = pg.unchecked_add(y, e);                 // 4 [pat[j] == 0] + #equal blocks  in [0, 8]
            ok.push_back(pg.pbs(y, [](uint64_t x) { return uint64_t(x >= 4); }));
        }
        return isk.are_all_comparisons_block_true(ok);
    }
    std::vector<Ct> zero_flags(const FheString &s) {
        std::vector<Ct> z;
        for (auto &c : s.chars) z.push_back(is_zero(c));
        return z;
    }
    BooleanBlock starts_with(const FheString &hay, const FheString &pat) {
        if (pat.len() == 0) return pg.create_trivial(1);
        return window_match(hay, pat, 0, zero_flags(pat));
    }
    BooleanBlock contains(const FheString &hay, const FheString &pat) {
        if (pat.len() == 0) return pg.create_trivial(1);
        std::vector<Ct> pz = zero_flags(pat), m;
        for (size_t w = 0; w < std::max<size_t>(hay.len(), 1); ++w) m.push_back(window_match(hay, pat, w, pz));
        return isk.is_at_least_one_comparisons_block_true(m);
    }
    // find / rfind with a padded pattern (str::find / str::rfind: byte index of the first / last match; the empty pattern matches at 0 and,
    // for rfind, at len).  Window w = 0 .. capacity: a match must start inside the string or right at its end (w == 0 or hay[w - 1] != 0),
    // which only matters for the empty pattern -- a non-empty one cannot match in the padding.  Index: radix digits of w, as string_find.
    std::pair<BooleanBlock, Radix> find(const FheString &hay, const FheString &pat, bool last) {
        const size_t n = hay.len();
        size_t idx_blocks = 1;
        while ((size_t(1) << (2 * idx_blocks)) < n + 1) ++idx_blocks;
        std::vector<Ct> pz = zero_flags(pat), m;
        for (size_t w = 0; w <= n; ++w) {
            Ct mw = w < n || pat.len() == 0 ? (pat.len() == 0 ? pg.create_trivial(1) : window_match(hay, pat, w, pz))
                                            : isk.are_all_comparisons_block_true(pz);            // w == n: only the empty pattern fits
            if (w > 0) mw = isk.boolean_bitand(mw, nonzero(hay.chars[w - 1]));
            m.push_back(mw);
        }
        if (last) std::reverse(m.begin(), m.end());
        return ssk.first_true(m, [=](size_t w) { return last ? n - w : w; }, idx_blocks);
    }

    // some suffix of the haystack equals the pattern as padded strings (the empty suffix included)
    BooleanBlock ends_with(const FheString &hay, const FheString &pat) { return isk.is_at_least_one_comparisons_block_true(suffix_matches(hay, pat)); }
    // per[w], w = 0 ..= capacity: hay[w..] equals the pattern as padded strings.  A non-empty pattern fires at w = len - len(pat) only, the
    // empty one at every w >= len
    std::vector<Ct> suffix_matches(const FheString &hay, const FheString &pat) {
        const size_t n = hay.len(), m = pat.len();
        std::vector<Ct> pz = zero_flags(pat), hz = zero_flags(hay), per;
        for (size_t w = 0; w <= n; ++w) {
            std::vector<Ct> flags;
            const size_t span = std::max(n - w, m);
            for (size_t j = 0; j < span; ++j) {
                const bool in_h = w + j < n, in_p = j < m;
                if (in_h && in_p) {
                    std::vector<Ct> eqs = isk.block_equalities(hay.chars[w + j], pat.chars[j]);
                    flags.insert(flags.end(), eqs.begin(), eqs.end());
                } else if (in_h) flags.push_back(hz[w + j]);
                else flags.push_back(pz[j]);
            }
            per.push_back(isk.are_all_comparisons_block_true(flags));
        }
        return per;
    }

    // ---- strip_prefix / strip_suffix with a PADDED pattern: (matched, string) ---------------------------------------------------------
    // prefix: a left shift by len(pat), every bit of the amount gated by the flag
    std::pair<BooleanBlock, FheString> strip_prefix(const FheString &s, const FheString &pat) {
        BooleanBlock flag = starts_with(s, pat);
        if (pat.len() == 0) return {flag, s};
        size_t n_bits = 1;
        while ((size_t(1) << n_bits) <= pat.len()) ++n_bits;
        std::vector<Ct> bits = bits_of(len(pat), n_bits);
        for (auto &b : bits) b = and_flags(b, flag);
        return {flag, shift(s, bits, true)};
    }
    // suffix: the chars at and after the window where the pattern is the suffix are dropped (the first such window for the empty pattern)
    std::pair<BooleanBlock, FheString> strip_suffix(const FheString &s, const FheString &pat) {
        const size_t n = s.len();
        std::vector<Ct> drop = prefix_or(suffix_matches(s, pat), true);
        FheString out = s;
        for (size_t i = 0; i < n; ++i) out.chars[i] = keep(s.chars[i], isk.boolean_bitnot(drop[i]));
        return {drop[n], out};
    }

    // ---- eq_ignore_case of two padded strings: the fused ASCII case fold of both (the padding byte folds to itself), then eq -----------
    BooleanBlock eq_ignore_case(const FheString &a, const FheString &b) { return eq(ssk.to_lowercase(a), ssk.to_lowercase(b)); }

    // ---- concat / repeat: the second operand moves right by the secret length of the first; the supports are disjoint, so the result is a
    // leveled sum of blocks -----------------------------------------------------------------------------------------------------------------------
    FheString concat(const FheString &a, const FheString &b) {
        const size_t na = a.len(), nb = b.len(), n = na + nb;
        if (na == 0) return b;
        if (nb == 0) return a;
        Radix la = len(a);
        size_t n_bits = 1;
        while ((size_t(1) << n_bits) <= na) ++n_bits;
        FheString bs = shift(extend(b, n), bits_of(la, n_bits), false);
        FheString ae = extend(a, n), out;
        for (size_t i = 0; i < n; ++i) {
            Radix c;
            for (size_t k = 0; k < 4; ++k) {
                Ct v = pg.unchecked_add(ae.chars[i][k], bs.chars[i][k]);
                v.degree = p.msg_mod - 1;        // at most one of the two blocks is non-zero
                c.push_back(v);
            }
            out.chars.push_back(c);
        }
        return out;
    }
    FheString repeat(const FheString &s, size_t count) {
        if (count == 0) { FheString e; return e; }
        FheString acc = s;
        for (size_t k = 1; k < count; ++k) acc = concat(acc, s);
        return acc;
    }
    // repeat by a secret count: s repeated min(count, max_count) times in capacity * max_count chars.  Copy k is s masked by
    // [k < count], and the copies are concatenated: an empty copy moves nothing.  Every concat adds one unit of noise to the chars it
    // keeps, so they are cleaned before len() would sum four blocks of more than 3 units, and at the end
    FheString repeat(const FheString &s, const Radix &count, size_t max_count) {
        FheString acc;
        if (max_count == 0) return acc;
        const Radix limit = clamp_radix(count, digits_for(max_count));
        for (size_t k = 0; k < max_count; ++k) {
            const Ct more = pg.pbs(scalar_sign(limit, k), [](uint64_t x) { return uint64_t(x == IntegerServerKey::IS_SUPERIOR); });
            FheString copy;
            for (auto &c : s.chars) copy.chars.push_back(keep(c, more));
            acc = k == 0 ? copy : concat(cleaned(acc, 3), copy);
        }
        return cleaned(acc, 1);
    }
    // every block of noise above max_noise through a message-extract PBS
    FheString cleaned(const FheString &s, uint64_t max_noise) {
        FheString out = s;
        for (auto &c : out.chars)
            for (auto &blk : c)
                if (blk.noise > max_noise || blk.degree >= p.msg_mod) blk = pg.pbs(blk, [this](uint64_t x) { return x % p.msg_mod; });
        return out;
    }

    // ---- replace / replacen / split / splitn / split_once / rsplit_once: str's methods with a &str pattern ------------------------------
    // Matches are found left to right and never overlap; the empty pattern matches at every char boundary 0 ..= len.  The pattern is a
    // padded string (secret length, maybe empty) or a clear one (trivial chars, no padding, so its least length m_min is its length).
    // The sizes are public bounds: at most M = max_matches(capacity, m_min) matches, so
    //   replacen returns capacity + min(count, M) * max(0, capacity_to - m_min) chars, and split returns M + 1 parts (splitn: at most n).
    // Every step is a wide level of independent PBS plus leveled sums; no PBS input exceeds 15 nominal noise units, and every result block
    // is a PBS output or trivial.
    struct Pattern {
        FheString chars;
        std::string text;      // the clear pattern
        bool clear = false;
        size_t min_len() const { return clear ? chars.len() : 0; }
    };
    Pattern padded_pattern(const FheString &pat) { Pattern pt; pt.chars = pat; return pt; }
    Pattern clear_pattern(const std::string &text) { Pattern pt; pt.chars = ssk.trivial_string(text); pt.text = text; pt.clear = true; return pt; }
    static size_t max_matches(size_t capacity, size_t m_min) { return m_min == 0 ? capacity + 1 : capacity / m_min; }

    bool is_const(const Ct &c, uint64_t v) const { return c.is_trivial() && c.body == v * p.delta(); }
    Ct and_flags(const Ct &a, const Ct &b) {
        if (is_const(a, 0) || is_const(b, 0)) return pg.create_trivial(0);
        if (a.is_trivial()) return b;
        if (b.is_trivial()) return a;
        return isk.boolean_bitand(a, b);
    }
    // a + b where at most one is non-zero (the sum's degree is `degree`)
    Ct add_disjoint(const Ct &a, const Ct &b, uint64_t degree) {
        if (is_const(a, 0)) return b;
        if (is_const(b, 0)) return a;
        Ct s = pg.unchecked_add(a, b);
        s.degree = degree;
        return s;
    }
    Ct keep_block(const Ct &blk, const Ct &flag) {
        if (is_const(blk, 0) || is_const(flag, 0)) return pg.create_trivial(0);
        if (flag.is_trivial()) return blk;
        return pg.pbs_bivariate(blk, flag, [](uint64_t v, uint64_t k) { return (k & 1) ? v : uint64_t(0); });
    }
    Radix keep(const Radix &c, const Ct &flag) {
        Radix r;
        for (auto &blk : c) r.push_back(keep_block(blk, flag));
        return r;
    }
    // the sum of flags of which at most one is set, its noise kept <= budget: the earliest-ready flags are summed (15 units at a time)
    // and cleaned first, which keeps the cleaning off the critical path of a chain
    Ct onehot_sum(std::vector<Ct> t, uint64_t budget) {
        t.erase(std::remove_if(t.begin(), t.end(), [this](const Ct &c) { return is_const(c, 0); }), t.end());
        if (t.empty()) return pg.create_trivial(0);
        const uint64_t cap = p.total_mod() - 1;
        for (;;) {
            uint64_t total = 0;
            for (auto &c : t) total += c.noise;
            if (total <= budget) break;
            std::stable_sort(t.begin(), t.end(), [](const Ct &a, const Ct &b) { return a.ready < b.ready; });
            size_t k = 0;
            uint64_t noise = 0;
            while (k < t.size() && noise + t[k].noise <= cap) noise += t[k++].noise;
            if (k == 0 || (k == 1 && t[0].noise <= 1)) throw std::logic_error("onehot_sum: a flag is too noisy");
            Ct sum = t[0];
            for (size_t j = 1; j < k; ++j) sum = pg.unchecked_add(sum, t[j]);
            t.erase(t.begin(), t.begin() + k);
            t.push_back(pg.pbs(sum, [](uint64_t x) { return uint64_t(x != 0); }));
        }
        Ct sum = t[0];
        for (size_t j = 1; j < t.size(); ++j) sum = pg.unchecked_add(sum, t[j]);
        sum.degree = 1;
        return sum;
    }
    // inclusive prefix counts of boolean flags, each a radix of nd digits: Hillis-Steele over the positions, one radix addition
    // (add_parallelized) per position and step, on only as many digits as the counts of that step can fill
    std::vector<Radix> prefix_count(const std::vector<Ct> &f, size_t nd) {
        const size_t n = f.size();
        std::vector<Radix> c(n);
        for (size_t i = 0; i < n; ++i) {
            c[i].push_back(f[i]);
            while (c[i].size() < nd) c[i].push_back(pg.create_trivial(0));
        }
        for (size_t d = 1; d < n; d *= 2) {
            const size_t used = std::min(nd, digits_for(std::min(2 * d, n)));
            std::vector<Radix> nxt = c;
            for (size_t i = d; i < n; ++i) {
                Radix s = isk.add(Radix(c[i].begin(), c[i].begin() + used), Radix(c[i - d].begin(), c[i - d].begin() + used));
                while (s.size() < nd) s.push_back(pg.create_trivial(0));
                nxt[i] = s;
            }
            c.swap(nxt);
        }
        return c;
    }
    // sign of (digits - c): 0 less, 1 equal, 2 greater.  Pairs of digits are compared with c by table lookup and the signs reduced with
    // the comparator's tree; nothing is subtracted, so no value reaches the padding bit
    Ct scalar_sign(const Radix &digits, uint64_t c) {
        std::vector<Ct> packed = isk.pack_pairs(digits), signs;
        for (size_t i = 0; i < packed.size(); ++i) {
            const uint64_t mod = 2 * i + 1 < digits.size() ? uint64_t(p.msg_mod) * p.msg_mod : p.msg_mod, cv = c % mod;
            c /= mod;
            signs.push_back(pg.pbs(packed[i], [cv](uint64_t x) { return x < cv ? uint64_t(0) : (x == cv ? uint64_t(1) : uint64_t(2)); }));
        }
        if (c != 0) return pg.create_trivial(IntegerServerKey::IS_INFERIOR);
        return isk.reduce_signs(signs);
    }
    Radix trivial_radix(uint64_t v, size_t nd) {
        Radix r;
        for (size_t b = 0; b < nd; ++b) r.push_back(pg.create_trivial((v >> (2 * b)) & 3));
        return r;
    }

    struct Matches {
        std::vector<Ct> raw;         // windows 0 ..= capacity: the pattern occurs at w (and w is inside the string or at its end)
        std::vector<Ct> over, cov;   // d = 0 .. cap_pat - 1: matches d apart can overlap (d >= 1) / a match covers the char d after its start
    };
    // hay_nz: where given, receives nonzero_flags(hay) when a padded pattern needs them (left untouched otherwise)
    Matches find_all(const FheString &hay, const Pattern &pt, std::vector<Ct> *hay_nz = nullptr) {
        const size_t n = hay.len(), m = pt.chars.len();
        Matches r;
        r.raw.assign(n + 1, pg.create_trivial(0));
        if (m == 0) {
            std::vector<Ct> nz = nonzero_flags(hay);
            r.raw[0] = pg.create_trivial(1);
            for (size_t w = 1; w <= n; ++w) r.raw[w] = nz[w - 1];
            return r;
        }
        if (pt.clear) {
            // a non-empty clear pattern starts with a non-zero char, so it never matches in the padding.  Two matches d apart can both be
            // candidates only if d is a period of the pattern (it has a border of length m - d); every other shift needs no check
            std::vector<Ct> mw = ssk.window_matches(hay, pt.chars);   // windows 0 ..= n - m
            for (size_t w = 0; w < mw.size(); ++w) r.raw[w] = mw[w];
            for (size_t d = 0; d < m; ++d) {
                r.cov.push_back(pg.create_trivial(1));
                r.over.push_back(pg.create_trivial(d > 0 && pt.text.compare(d, m - d, pt.text, 0, m - d) == 0));
            }
            return r;
        }
        // padded: as find -- a window must start inside the string or right at its end, which only matters for the empty pattern
        std::vector<Ct> pz = zero_flags(pt.chars), nz = nonzero_flags(hay);
        for (size_t w = 0; w <= n; ++w) {
            Ct mw = w < n ? window_match(hay, pt.chars, w, pz) : isk.are_all_comparisons_block_true(pz);
            r.raw[w] = w > 0 ? isk.boolean_bitand(mw, nz[w - 1]) : mw;
        }
        if (hay_nz) *hay_nz = nz;
        for (size_t d = 0; d < m; ++d) r.cov.push_back(isk.boolean_bitnot(pz[d]));   // [the pattern is longer than d]
        r.over = r.cov;
        return r;
    }
    // leftmost non-overlapping matches: acc[w] = raw[w] AND NOT OR_{1 <= d < cap_pat} (acc[w - d] AND over[d]).  A chain over w where some
    // over[d] can be set; with a clear pattern that has no proper border every over[d] is trivially 0 and acc = raw.
    std::vector<Ct> non_overlapping(const std::vector<Ct> &raw, const std::vector<Ct> &over) {
        std::vector<Ct> acc(raw.size());
        for (size_t w = 0; w < raw.size(); ++w) {
            acc[w] = raw[w];
            if (is_const(raw[w], 0)) continue;
            std::vector<Ct> t;
            for (size_t d = 1; d < over.size() && d <= w; ++d) t.push_back(and_flags(acc[w - d], over[d]));
            Ct blocked = onehot_sum(t, p.total_mod() - 1 - raw[w].noise);   // at most one accepted match covers w
            if (is_const(blocked, 0)) continue;
            acc[w] = pg.pbs(pg.unchecked_add(isk.boolean_bitnot(raw[w]), blocked), [](uint64_t x) { return uint64_t(x == 0); });
        }
        return acc;
    }
    // covered[i] = OR_d (starts[i - d] AND cov[d]) for the chars i < n; the starts never overlap, so this is a sum (noise <= 2)
    std::vector<Ct> covered(const std::vector<Ct> &starts, const std::vector<Ct> &cov, size_t n) {
        std::vector<Ct> out(n);
        for (size_t i = 0; i < n; ++i) {
            std::vector<Ct> t;
            for (size_t d = 0; d < cov.size() && d <= i; ++d) t.push_back(and_flags(starts[i - d], cov[d]));
            out[i] = onehot_sum(t, 2);
        }
        return out;
    }
    // the first `limit` of the accepted matches: acc[w] AND [count of accepted matches up to w <= limit]
    std::vector<Ct> first_matches(const std::vector<Ct> &acc, const std::vector<Radix> &cnt, size_t limit) {
        std::vector<Ct> lim(acc.size());
        for (size_t w = 0; w < acc.size(); ++w)
            lim[w] = is_const(acc[w], 0) ? acc[w]
                                         : pg.pbs_bivariate(scalar_sign(cnt[w], limit), acc[w], [](uint64_t s, uint64_t a) { return uint64_t(s != 2 && (a & 1)); });
        return lim;
    }

    // ---- secret integer arguments: a radix of any number of digits, little endian ---------------------------------------------------
    // the low nd digits, zero-extended, or all maximal when a higher digit is set: min(x, 4^nd - 1), so one comparison on nd digits decides
    Radix clamp_radix(const Radix &x, size_t nd) {
        Radix lo = resized(Radix(x.begin(), x.begin() + std::min(nd, x.size())), nd);
        if (x.size() <= nd) return lo;
        std::vector<Ct> high;
        for (size_t j = nd; j < x.size(); ++j) high.push_back(pg.pbs(x[j], [](uint64_t v) { return uint64_t(v != 0); }));
        const Ct over = isk.is_at_least_one_comparisons_block_true(high);
        const uint64_t top = p.msg_mod - 1;
        for (auto &d : lo) d = pg.pbs_bivariate(d, over, [top](uint64_t v, uint64_t o) { return (o & 1) ? top : v; });
        return lo;
    }
    // sign of (a - b) for radixes of the same length: block signs by bivariate lookup, reduced with the comparator's tree; as in
    // scalar_sign nothing is subtracted
    Ct radix_sign(const Radix &a, const Radix &b) {
        std::vector<Ct> signs;
        for (size_t i = 0; i < a.size(); ++i)
            signs.push_back(pg.pbs_bivariate(a[i], b[i], [](uint64_t x, uint64_t y) {
                return x < y ? IntegerServerKey::IS_INFERIOR : (x == y ? IntegerServerKey::IS_EQUAL : IntegerServerKey::IS_SUPERIOR);
            }));
        return isk.reduce_signs(signs);
    }
    Radix resized(Radix r, size_t nd) {
        while (r.size() < nd) r.push_back(pg.create_trivial(0));
        r.resize(nd);
        return r;
    }
    // first_matches with a secret limit (at least as many digits as the counts): acc[w] AND [cnt[w] < limit] (strict) or [cnt[w] <= limit]
    std::vector<Ct> first_matches_below(const std::vector<Ct> &acc, const std::vector<Radix> &cnt, const Radix &limit, bool strict) {
        std::vector<Ct> lim(acc.size());
        for (size_t w = 0; w < acc.size(); ++w) {
            if (is_const(acc[w], 0)) { lim[w] = acc[w]; continue; }
            const Ct sign = radix_sign(resized(cnt[w], limit.size()), limit);
            lim[w] = pg.pbs_bivariate(sign, acc[w], [strict](uint64_t s, uint64_t a) {
                return uint64_t((strict ? s == IntegerServerKey::IS_INFERIOR : s != IntegerServerKey::IS_SUPERIOR) && (a & 1));
            });
        }
        return lim;
    }

    // ends[e], e = 0 ..= capacity: one of the matches `starts` (window order, non-overlapping) ends at e.  A clear pattern of length m:
    // starts[e - m].  A padded one: OR_d (starts[e - d] AND [len(pat) == d]); one length is true, so the terms are disjoint (built as
    // `covered` is)
    std::vector<Ct> match_ends(const std::vector<Ct> &starts, const Pattern &pt) {
        const size_t n = starts.size() - 1, m = pt.chars.len();
        std::vector<Ct> ends(n + 1, pg.create_trivial(0));
        if (pt.clear) {
            for (size_t e = m; e <= n; ++e) ends[e] = starts[e - m];
            return ends;
        }
        const std::vector<Ct> is_len = length_onehot(nonzero_flags(pt.chars));   // d = 0 ..= cap_pat
        for (size_t e = 0; e <= n; ++e) {
            std::vector<Ct> t;
            for (size_t d = 0; d <= std::min(e, m); ++d) t.push_back(and_flags(starts[e - d], is_len[d]));
            ends[e] = onehot_sum(t, 1);
        }
        return ends;
    }
    // [the part at the end of the string is empty]: the string is empty, or one of the matches ends at its end
    Ct end_part_empty(const FheString &s, const std::vector<Ct> &ends) {
        const std::vector<Ct> at_len = length_onehot(nonzero_flags(s));
        std::vector<Ct> t{at_len[0]};
        for (size_t e = 1; e <= s.len(); ++e) t.push_back(and_flags(at_len[e], ends[e]));
        return onehot_sum(t, 1);
    }

    // removes the zero chars of s in order and returns the first out_len positions.  Char j moves left by the number D_j of zero chars
    // before it, one bit of D_j per stage, least significant first.  For non-zero chars j < j', D_j' - D_j <= j' - j - 1, so their
    // positions stay strictly increasing after every stage: no two chars ever meet, a stage is a sum of two keep_if per block, and the
    // remaining bits of D_j travel with their char.
    FheString compact(const FheString &s, size_t out_len) {
        const size_t E = s.len();
        FheString out;
        if (E == 0) return extend(out, out_len);
        std::vector<Ct> z(E);
        for (size_t j = 0; j < E; ++j) z[j] = is_zero(s.chars[j]);
        size_t T = 0;
        while ((size_t(1) << T) <= E - 1) ++T;
        std::vector<Radix> D = prefix_count(z, digits_for(E));
        std::vector<std::vector<Ct>> B(T, std::vector<Ct>(E));
        for (size_t t = 0; t < T; ++t)
            for (size_t j = 0; j < E; ++j)
                B[t][j] = pg.pbs_bivariate(D[j][t / 2], z[j], [t](uint64_t d, uint64_t zz) { return (zz & 1) ? uint64_t(0) : (d >> (t % 2)) & 1; });
        FheString cur = s;
        for (size_t t = 0; t < T; ++t) {
            const size_t k = size_t(1) << t, reach = (size_t(1) << T) - (size_t(2) << t);   // what the later stages can still move a char
            const size_t live = std::min(E, out_len + reach);
            FheString nxt;
            nxt.chars.assign(E, trivial_char(0));
            std::vector<std::vector<Ct>> nB(T, std::vector<Ct>(E, pg.create_trivial(0)));
            for (size_t i = 0; i < live; ++i) {
                const Ct stay = isk.boolean_bitnot(B[t][i]);
                const bool src = i + k < E;
                const Ct zero = pg.create_trivial(0), move = src ? B[t][i + k] : zero;
                for (size_t b = 0; b < 4; ++b)
                    nxt.chars[i][b] = add_disjoint(keep_block(cur.chars[i][b], stay), src ? keep_block(cur.chars[i + k][b], move) : zero, p.msg_mod - 1);
                for (size_t u = t + 1; u < T; ++u)
                    nB[u][i] = add_disjoint(and_flags(B[u][i], stay), src ? and_flags(B[u][i + k], move) : zero, 1);
            }
            cur = nxt;
            B = nB;
        }
        for (size_t i = 0; i < std::min(out_len, E); ++i) {
            Radix c;
            for (auto &blk : cur.chars[i])
                c.push_back(blk.noise <= 1 && blk.degree < p.msg_mod ? blk : pg.pbs(blk, [this](uint64_t x) { return x % p.msg_mod; }));
            out.chars.push_back(c);
        }
        return extend(out, out_len);
    }

    // replacen (count = SIZE_MAX: replace; secret_count: the first *secret_count matches, sized as replace).  Slot i of the expanded string
    // holds `to` if an accepted match starts at i, then s[i] unless a match covers it; compacting the zero chars away gives the result
    FheString replace(const FheString &s, const Pattern &pt, const FheString &to, size_t count, const Radix *secret_count = nullptr) {
        const size_t n = s.len(), m_min = pt.min_len(), M = max_matches(n, m_min);
        count = std::min(count, M);
        const size_t out_len = n + count * (to.len() > m_min ? to.len() - m_min : 0);
        if (count == 0) return s;
        Matches mt = find_all(s, pt);
        std::vector<Ct> acc = non_overlapping(mt.raw, mt.over);
        if (secret_count) {
            std::vector<Radix> cnt = prefix_count(acc, digits_for(M));
            acc = first_matches_below(acc, cnt, clamp_radix(*secret_count, digits_for(M)), false);
        } else if (count < M) acc = first_matches(acc, prefix_count(acc, digits_for(M)), count);
        std::vector<Ct> cov = covered(acc, mt.cov, n);
        FheString ex;   // chars known to be zero are left out: compaction removes them anyway
        for (size_t i = 0; i <= n; ++i) {
            if (!is_const(acc[i], 0))
                for (auto &c : to.chars) ex.chars.push_back(keep(c, acc[i]));
            if (i < n && !is_const(cov[i], 1)) ex.chars.push_back(keep(s.chars[i], isk.boolean_bitnot(cov[i])));
        }
        return compact(ex, out_len);
    }

    // the chars of s selected by `in` -- one contiguous run, which may reach into the padding -- moved to the start
    FheString part(const FheString &s, const std::vector<Ct> &in) {
        const size_t n = s.len();
        FheString masked;
        for (size_t i = 0; i < n; ++i) masked.chars.push_back(keep(s.chars[i], in[i]));
        if (n <= 1) return masked;
        std::vector<Ct> st(n);   // one-hot: the run starts at i
        st[0] = in[0];
        for (size_t i = 1; i < n; ++i)
            st[i] = pg.pbs(pg.unchecked_add(in[i], pg.unchecked_scalar_mul(in[i - 1], 2)), [](uint64_t x) { return uint64_t(x == 1); });
        size_t n_bits = 0;
        while ((size_t(1) << n_bits) <= n - 1) ++n_bits;
        Radix start = onehot_to_radix(st, digits_for(n - 1), [](size_t w) { return uint64_t(w); });
        return shift(masked, bits_of(start, n_bits), true);
    }

    // splitn (n_parts = SIZE_MAX: split): (part count as digits_for(P) digits, P parts of capacity chars), P = min(M + 1, n_parts).  Char i
    // belongs to part min(#accepted matches at or before i, P - 1) unless a match covers it; parts past the count are empty.
    //   reverse      rsplit / rsplitn: the rightmost non-overlapping matches (the reverse searcher: the chain runs from window `capacity`
    //                down), and char i belongs to part #accepted matches after i, part 0 being the one at the end of the string
    //   terminator   split_terminator / rsplit_terminator: the part at the end of the string is dropped when it is empty.  For split that
    //                is the last part, which is then all zero already, so only the count drops; for rsplit it is part 0, so every char's
    //                part index drops by that flag
    //   secret_n     splitn_enc / rsplitn_enc: n is a radix, P = M + 1; the first n - 1 matches split, part n - 1 is the unsplit rest
    std::pair<Radix, std::vector<FheString>> split(const FheString &s, const Pattern &pt, size_t n_parts, bool reverse = false,
                                                   bool terminator = false, const Radix *secret_n = nullptr) {
        const size_t n = s.len(), M = max_matches(n, pt.min_len()), P = std::min(M + 1, n_parts), nd = digits_for(P);
        std::vector<FheString> parts;
        if (P == 0) return {trivial_radix(0, nd), parts};
        if (P == 1 && !terminator && !secret_n) { parts.push_back(s); return {trivial_radix(1, nd), parts}; }
        const size_t last = P - 1;
        Matches mt = find_all(s, pt);
        std::vector<Ct> raw = mt.raw;                                 // in the order the searcher meets the windows
        if (reverse) std::reverse(raw.begin(), raw.end());
        std::vector<Ct> acc = non_overlapping(raw, mt.over);
        std::vector<Radix> cnt = prefix_count(acc, digits_for(M));   // counts of every accepted match, up to M
        const Radix limit = secret_n ? clamp_radix(*secret_n, nd) : Radix();
        std::vector<Ct> lim = secret_n ? first_matches_below(acc, cnt, limit, true) : last < M ? first_matches(acc, cnt, last) : acc;
        if (reverse) std::reverse(lim.begin(), lim.end());           // back to window order
        std::vector<Ct> cov = covered(lim, mt.cov, n);
        // matches before char i in the searcher's order: at or before i, or (reverse) after i
        auto count_at = [&](size_t i) -> const Radix & { return cnt[reverse ? n - 1 - i : i]; };
        // count = min(#matches, last) + 1: when there are fewer than `last` matches, their number fits nd digits
        Radix total(cnt[n].begin(), cnt[n].begin() + std::min(nd, cnt[n].size()));
        while (total.size() < nd) total.push_back(pg.create_trivial(0));
        Radix count;
        Ct dropped;                                                    // terminator: the part at the end is empty
        if (terminator) {
            dropped = end_part_empty(s, match_ends(lim, pt));
            count = isk.add(total, resized({isk.boolean_bitnot(dropped)}, nd));
        } else count = isk.add(total, trivial_radix(1, nd));
        if (secret_n) {                                                // min(#matches + 1, n)
            Ct less = pg.pbs(radix_sign(count, limit), [](uint64_t x) { return uint64_t(x == IntegerServerKey::IS_INFERIOR); });
            count = isk.if_then_else(less, count, limit);
        } else if (last < M) {
            Ct more = pg.pbs(scalar_sign(cnt[n], last), [](uint64_t x) { return uint64_t(x != 0); });
            count = isk.if_then_else(more, trivial_radix(P, nd), count);
        }
        // member(k, i): char i is in part k (of split / rsplit / splitn / rsplitn); in_part(k)[i]: char i goes to part k of the result
        auto member = [&](size_t k, size_t i) {
            const bool tail = k == last;
            return pg.pbs_bivariate(scalar_sign(count_at(i), k), cov[i], [tail](uint64_t sg, uint64_t c) {
                return uint64_t((tail ? sg != 0 : sg == 1) && !(c & 1));
            });
        };
        std::vector<std::vector<Ct>> members;                         // rsplit_terminator: [char i is in rsplit's part k], every k
        if (reverse && terminator)
            for (size_t k = 0; k < P; ++k) {
                members.emplace_back(n);
                for (size_t i = 0; i < n; ++i) members[k][i] = member(k, i);
            }
        std::vector<Ct> n_sign(P);                                     // secret n: sign of n - (k + 1)
        if (secret_n)
            for (size_t k = 0; k < P; ++k) n_sign[k] = scalar_sign(limit, k + 1);
        auto in_part = [&](size_t k) {
            std::vector<Ct> in(n);
            for (size_t i = 0; i < n; ++i) {
                if (reverse && terminator) {                           // part k of the result is rsplit's part k + dropped
                    const Ct next = k + 1 < P ? members[k + 1][i] : pg.create_trivial(0);
                    in[i] = pg.pbs_bivariate(pg.unchecked_add(members[k][i], pg.unchecked_scalar_mul(next, 2)), dropped,
                                             [](uint64_t x, uint64_t d) { return (d & 1) ? (x >> 1) & 1 : x & 1; });
                } else if (secret_n) {                                 // [cnt == k and k < n - 1] or [cnt >= k and k == n - 1]
                    Ct g = pg.pbs(pg.unchecked_add(scalar_sign(count_at(i), k), pg.unchecked_scalar_mul(n_sign[k], 3)), [](uint64_t x) {
                        const uint64_t sg = x % 3, ns = x / 3;
                        return uint64_t((ns == IntegerServerKey::IS_SUPERIOR && sg == IntegerServerKey::IS_EQUAL) ||
                                        (ns == IntegerServerKey::IS_EQUAL && sg != IntegerServerKey::IS_INFERIOR));
                    });
                    in[i] = pg.pbs_bivariate(g, cov[i], [](uint64_t x, uint64_t c) { return uint64_t((x & 1) && !(c & 1)); });
                } else in[i] = member(k, i);
            }
            return in;
        };
        for (size_t k = 0; k < P; ++k) {
            std::vector<Ct> in = in_part(k);
            if (k == 0 && !reverse) {   // part 0 starts at 0
                FheString p0;
                for (size_t i = 0; i < n; ++i) p0.chars.push_back(keep(s.chars[i], in[i]));
                parts.push_back(p0);
            } else parts.push_back(part(s, in));
        }
        return {count, parts};
    }

    // split_inclusive: the leftmost matches, each part keeping the match that ends it, and a trailing empty part dropped.  Char i belongs to
    // part #matches ending at or before i (covered chars included); count = #matches + [the part at the end is not empty]; P = M + 1.
    std::pair<Radix, std::vector<FheString>> split_inclusive(const FheString &s, const Pattern &pt) {
        const size_t n = s.len(), M = max_matches(n, pt.min_len()), P = M + 1, nd = digits_for(P);
        Matches mt = find_all(s, pt);
        const std::vector<Ct> ends = match_ends(non_overlapping(mt.raw, mt.over), pt);
        std::vector<Radix> cnt = prefix_count(ends, digits_for(M));
        const Ct trailing = isk.boolean_bitnot(end_part_empty(s, ends));
        Radix count = isk.add(resized(cnt[n], nd), resized({trailing}, nd));
        std::vector<FheString> parts;
        for (size_t k = 0; k < P; ++k) {
            std::vector<Ct> in(n);
            for (size_t i = 0; i < n; ++i)
                in[i] = pg.pbs(scalar_sign(cnt[i], k), [](uint64_t x) { return uint64_t(x == IntegerServerKey::IS_EQUAL); });
            if (k == 0) {   // part 0 starts at 0
                FheString p0;
                for (size_t i = 0; i < n; ++i) p0.chars.push_back(keep(s.chars[i], in[i]));
                parts.push_back(p0);
            } else parts.push_back(part(s, in));
        }
        return {count, parts};
    }

    // split_ascii_whitespace: the non-empty runs of chars that are neither padding nor u8::is_ascii_whitespace (U+0009, U+000A, U+000C,
    // U+000D, U+0020 -- not U+000B, which char::is_whitespace and char_class include).  Word k holds the chars after the (k + 1)-th word
    // start; P = ceil(capacity / 2) parts.
    Ct ascii_word_char(const Radix &c) {
        Ct hi = pg.unchecked_add(pg.unchecked_scalar_mul(c[3], p.msg_mod), c[2]);
        Ct lo = pg.unchecked_add(pg.unchecked_scalar_mul(c[1], p.msg_mod), c[0]);
        Ct k = pg.pbs(hi, [](uint64_t x) { return x == 0 ? uint64_t(1) : (x == 2 ? uint64_t(2) : uint64_t(0)); });
        Ct r = pg.pbs(lo, [](uint64_t x) { return x == 0 ? uint64_t(2) : ((x == 9 || x == 10 || x == 12 || x == 13) ? uint64_t(1) : uint64_t(0)); });
        return pg.pbs_bivariate(k, r, [](uint64_t kk, uint64_t rr) {
            return uint64_t(!((kk == 1 && rr != 0) || (kk == 2 && rr == 2)));   // 0x00, 0x09, 0x0A, 0x0C, 0x0D, 0x20
        });
    }
    std::pair<Radix, std::vector<FheString>> split_ascii_whitespace(const FheString &s) {
        if (s.len() == 0) return words(s, {});
        std::vector<Ct> word(s.len());
        for (size_t i = 0; i < s.len(); ++i) word[i] = ascii_word_char(s.chars[i]);
        return words(s, word);
    }
    // the words of s given the flags [char i is a word char] (padding is not): count, then P = ceil(capacity / 2) words
    std::pair<Radix, std::vector<FheString>> words(const FheString &s, const std::vector<Ct> &word) {
        const size_t n = s.len(), P = (n + 1) / 2, nd = digits_for(P);
        std::vector<FheString> parts;
        if (n == 0) return {trivial_radix(0, nd), parts};
        std::vector<Ct> start(n);
        start[0] = word[0];
        for (size_t i = 1; i < n; ++i)
            start[i] = pg.pbs(pg.unchecked_add(word[i], pg.unchecked_scalar_mul(word[i - 1], 2)), [](uint64_t x) { return uint64_t(x == 1); });
        std::vector<Radix> cnt = prefix_count(start, nd);
        for (size_t k = 0; k < P; ++k) {
            std::vector<Ct> in(n);
            for (size_t i = 0; i < n; ++i)
                in[i] = pg.pbs_bivariate(scalar_sign(cnt[i], k + 1), word[i], [](uint64_t sg, uint64_t w) { return uint64_t(sg == IntegerServerKey::IS_EQUAL && (w & 1)); });
            parts.push_back(part(s, in));
        }
        return {cnt[n - 1], parts};
    }

    // split_once / rsplit_once: (found, before, after) around the first (last: the last, as rfind finds it) match; both strings are empty
    // when there is none
    std::tuple<BooleanBlock, FheString, FheString> split_once(const FheString &s, const Pattern &pt, bool last) {
        const size_t n = s.len();
        Matches mt = find_all(s, pt);
        std::vector<Ct> raw = mt.raw;
        if (last) std::reverse(raw.begin(), raw.end());
        std::vector<Ct> any = prefix_or(raw, true);   // [a match at or before w] (last: at or after w)
        if (last) std::reverse(any.begin(), any.end());
        auto flag_sub = [this](const Ct &a, const Ct &b) { Ct r = pg.lwe_sub(a, b); r.degree = 1; return r; };
        const Ct found = last ? any[0] : any[n];
        std::vector<Ct> start(n + 1);                  // one-hot: the splitting match
        for (size_t w = 0; w <= n; ++w) {
            if (last) start[w] = w < n ? flag_sub(any[w], any[w + 1]) : any[n];
            else start[w] = w > 0 ? flag_sub(any[w], any[w - 1]) : any[0];
        }
        std::vector<Ct> cov = covered(start, mt.cov, n), before(n), after(n);
        for (size_t i = 0; i < n; ++i) {
            before[i] = last ? any[i + 1] : flag_sub(found, any[i]);
            after[i] = last ? flag_sub(flag_sub(found, any[i + 1]), cov[i]) : flag_sub(any[i], cov[i]);
        }
        FheString b;
        for (size_t i = 0; i < n; ++i) b.chars.push_back(keep(s.chars[i], before[i]));
        return {found, b, part(s, after)};
    }

    // ---- matches / match_indices / rmatch_indices / trim_start_matches / trim_end_matches: the rest of str's &str-pattern methods ------
    // matches(pat) always yields the pattern itself, so its iterator carries only a count.  There is no separate rmatches count: with
    // every match of one length, greedy selection from the left and from the right both find a largest set of non-overlapping matches,
    // so the two counts are equal (the empty pattern: len + 1 either way).
    // the number of set flags as nd digits (a tree of radix additions, each on as many digits as its partial sums can fill)
    Radix count_flags(const std::vector<Ct> &f, size_t nd) {
        std::vector<std::pair<Radix, size_t>> c;   // partial sums and their largest value
        for (auto &x : f)
            if (!is_const(x, 0)) c.push_back({Radix{x}, 1});
        if (c.empty()) return trivial_radix(0, nd);
        while (c.size() > 1) {
            std::vector<std::pair<Radix, size_t>> nxt;
            for (size_t i = 0; i + 1 < c.size(); i += 2) {
                const size_t bound = c[i].second + c[i + 1].second, used = std::min(nd, digits_for(bound));
                nxt.push_back({isk.add(resized(c[i].first, used), resized(c[i + 1].first, used)), bound});
            }
            if (c.size() % 2) nxt.push_back(c.back());
            c.swap(nxt);
        }
        return resized(c[0].first, nd);
    }
    // s.matches(pat).count(), digits_for(M) digits
    Radix matches(const FheString &s, const Pattern &pt) {
        const size_t M = max_matches(s.len(), pt.min_len());
        if (M == 0) return trivial_radix(0, 1);
        Matches mt = find_all(s, pt);
        return count_flags(non_overlapping(mt.raw, mt.over), digits_for(M));
    }
    // (count, M byte indices of digits_for(capacity) digits): the leftmost non-overlapping matches in order, or (reverse) the rightmost
    // ones from the end, as rsplit's reverse searcher finds them.  Index k is the window w with acc[w] and cnt[w] == k + 1 (in the
    // searcher's order), its radix the window's byte index; indices past the count are zero
    std::pair<Radix, std::vector<Radix>> match_indices(const FheString &s, const Pattern &pt, bool reverse) {
        const size_t n = s.len(), m_min = pt.min_len(), M = max_matches(n, m_min), nd = digits_for(M), ni = digits_for(n);
        std::vector<Radix> idx;
        if (M == 0) return {trivial_radix(0, nd), idx};
        Matches mt = find_all(s, pt);
        std::vector<Ct> raw = mt.raw;                                // in the order the searcher meets the windows
        if (reverse) std::reverse(raw.begin(), raw.end());
        const std::vector<Ct> acc = non_overlapping(raw, mt.over);
        const std::vector<Radix> cnt = prefix_count(acc, nd);
        for (size_t k = 0; k < M; ++k) {
            std::vector<Ct> sel(n + 1, pg.create_trivial(0));
            for (size_t r = 0; r <= n; ++r) {
                // matches are at least m_min apart: at most r / m_min + 1 of them (r + 1 for m_min = 0) up to the r-th window
                if (is_const(acc[r], 0) || k > (m_min ? r / m_min : r)) continue;
                sel[r] = pg.pbs_bivariate(scalar_sign(cnt[r], k + 1), acc[r], [](uint64_t sg, uint64_t a) {
                    return uint64_t(sg == IntegerServerKey::IS_EQUAL && (a & 1));
                });
            }
            idx.push_back(onehot_to_radix(sel, ni, [=](size_t r) { return uint64_t(reverse ? n - r : r); }));
        }
        return {cnt[n], idx};
    }
    // [len(pat) == d], d = 0 ..= capacity_pat, of a padded pattern
    std::vector<Ct> pattern_length_onehot(const Pattern &pt) { return length_onehot(nonzero_flags(pt.chars)); }
    // trim_start_matches: the run of back-to-back matches at the start goes (next_reject).  For a pattern length d the run covers chars
    // i < d j_d, j_d the first window 0, d, 2 d, ... that does not match; a padded pattern computes every d = 1 ..= capacity_pat and
    // selects with [len(pat) == d], so no chain over the string is needed.  The rest moves to the start in one `part`
    FheString trim_start_matches(const FheString &s, const Pattern &pt) {
        const size_t n = s.len(), m = pt.chars.len();
        if (m == 0 || (pt.clear && m > n)) return s;   // the empty pattern, or no match fits
        std::vector<Ct> raw(n + 1, pg.create_trivial(0)), is_len;
        if (pt.clear)   // only the windows at multiples of m
            for (size_t w = 0; w + m <= n; w += m) raw[w] = ssk.window_matches(s, pt.chars, w, w + 1)[0];
        else {
            raw = find_all(s, pt).raw;
            is_len = pattern_length_onehot(pt);
        }
        std::vector<std::vector<Ct>> terms(n);          // [char i is in the run] for each candidate length: at most one is set
        for (size_t d = pt.clear ? m : 1; d <= m && d <= n; ++d) {
            std::vector<Ct> fail;
            for (size_t w = 0; w + d <= n; w += d) fail.push_back(isk.boolean_bitnot(raw[w]));
            const std::vector<Ct> broken = prefix_or(fail, true);    // some window 0, d, ..., j d does not match
            const Ct sel = pt.clear ? pg.create_trivial(1) : is_len[d];
            for (size_t i = 0; i < fail.size() * d; ++i) terms[i].push_back(and_flags(sel, isk.boolean_bitnot(broken[i / d])));
        }
        std::vector<Ct> in(n);
        for (size_t i = 0; i < n; ++i) in[i] = isk.boolean_bitnot(onehot_sum(terms[i], 5));   // part() adds 3 in[]: <= 15
        return part(s, in);
    }
    // trim_end_matches: the run of back-to-back matches that ends at the secret end of the string goes (next_reject_back).  For a
    // pattern length d the run consists of the windows w = len - d, len - 2 d, ... down to the first that does not match.  Char i lies in
    // the window w_r(i) = the largest w <= i with w == r (mod d), r = len mod d, and goes iff no window w' >= w_r(i) of that residue class
    // below len fails: a suffix OR over the class, with one term per residue selected by [len == r (mod d)] (from length_onehot) and, for
    // a padded pattern, by [len(pat) == d].  Only a suffix is masked; nothing moves
    FheString trim_end_matches(const FheString &s, const Pattern &pt) {
        const size_t n = s.len(), m = pt.chars.len();
        if (m == 0 || (pt.clear && m > n)) return s;
        std::vector<Ct> nz, is_len;
        const std::vector<Ct> raw = find_all(s, pt, &nz).raw;
        if (pt.clear) nz = nonzero_flags(s);
        else is_len = pattern_length_onehot(pt);
        const std::vector<Ct> at_len = length_onehot(nz);
        std::vector<Ct> fail(n);                        // [w < len and no match at w]
        for (size_t w = 0; w < n; ++w)
            fail[w] = is_const(raw[w], 0) ? nz[w] : pg.pbs_bivariate(raw[w], nz[w], [](uint64_t r, uint64_t z) { return uint64_t(!(r & 1) && (z & 1)); });
        std::vector<std::vector<Ct>> terms(n);          // at most one term per char is set: one length, one residue
        for (size_t d = pt.clear ? m : 1; d <= m && d <= n; ++d) {
            const Ct sel = pt.clear ? pg.create_trivial(1) : is_len[d];
            for (size_t r = 0; r < d; ++r) {
                std::vector<Ct> t;
                for (size_t e = r; e <= n; e += d) t.push_back(at_len[e]);
                const Ct res = and_flags(sel, onehot_sum(t, 1));           // [len(pat) == d and len == r (mod d)]
                if (is_const(res, 0)) continue;
                std::vector<Ct> chain;                                     // the windows r, r + d, ... < n, last first
                for (size_t w = r; w < n; w += d) chain.push_back(fail[w]);
                std::reverse(chain.begin(), chain.end());
                std::vector<Ct> bad = prefix_or(chain, true);             // some failure at or after the window
                std::reverse(bad.begin(), bad.end());
                for (size_t i = r; i < n; ++i) terms[i].push_back(and_flags(res, isk.boolean_bitnot(bad[(i - r) / d])));
            }
        }
        FheString out = s;
        for (size_t i = 0; i < n; ++i) out.chars[i] = keep(s.chars[i], isk.boolean_bitnot(onehot_sum(terms[i], p.total_mod() - 1 - 4)));
        return out;
    }

    // ---- lines / split_whitespace -------------------------------------------------------------------------------------------------
    // a property of the byte c as one table lookup on hcode(high nibble) * mul + lcode(low nibble), given the two nibble codes (PBS
    // outputs).  The table is derived from the property over all 256 bytes; two bytes it tells apart must differ in their codes
    Ct byte_lookup(const Ct &hc, const Ct &lc, uint64_t mul, uint64_t (*hcode)(uint64_t), uint64_t (*lcode)(uint64_t), uint64_t (*prop)(uint64_t)) {
        std::vector<int> table(p.total_mod(), -1);
        for (uint64_t b = 0; b < 256; ++b) {
            const uint64_t x = hcode(b >> 4) * mul + lcode(b & 15), v = prop(b);
            if (x >= table.size() || (table[x] >= 0 && uint64_t(table[x]) != v)) throw std::logic_error("byte_lookup: the nibble codes do not separate the property");
            table[x] = int(v);
        }
        return pg.pbs(pg.unchecked_add(pg.unchecked_scalar_mul(hc, mul), lc), [table](uint64_t x) { return uint64_t(std::max(table[x], 0)); });
    }
    Ct high_nibble(const Radix &c) { return pg.unchecked_add(pg.unchecked_scalar_mul(c[3], p.msg_mod), c[2]); }
    Ct low_nibble(const Radix &c) { return pg.unchecked_add(pg.unchecked_scalar_mul(c[1], p.msg_mod), c[0]); }
    Ct nibble_code(const Ct &nib, uint64_t (*code)(uint64_t)) { return pg.pbs(nib, [code](uint64_t x) { return code(x); }); }

    // lines: split_inclusive on "\n", then a trailing "\n" or "\r\n" stripped from each line (a bare "\r" at the end stays).  Char i
    // belongs to line #("\n" before i) unless it is a "\n" or the "\r" of a "\r\n"; count = #"\n" + [the part at the end is not empty].
    // (count as digits_for(capacity) digits, capacity lines of capacity chars)
    std::pair<Radix, std::vector<FheString>> lines(const FheString &s) {
        const size_t n = s.len(), nd = digits_for(n);
        std::vector<FheString> parts;
        if (n == 0) return {trivial_radix(0, nd), parts};
        static uint64_t (*const h0)(uint64_t) = [](uint64_t h) { return uint64_t(h == 0); };
        static uint64_t (*const lnr)(uint64_t) = [](uint64_t l) { return l == 0xA ? uint64_t(1) : (l == 0xD ? uint64_t(2) : uint64_t(0)); };
        std::vector<Ct> nl(n), cr(n);
        for (size_t i = 0; i < n; ++i) {
            const Ct hc = nibble_code(high_nibble(s.chars[i]), h0), lc = nibble_code(low_nibble(s.chars[i]), lnr);
            nl[i] = byte_lookup(hc, lc, 3, h0, lnr, [](uint64_t b) { return uint64_t(b == '\n'); });
            cr[i] = byte_lookup(hc, lc, 3, h0, lnr, [](uint64_t b) { return uint64_t(b == '\r'); });
        }
        std::vector<Ct> in_line(n), ends(n + 1, pg.create_trivial(0));
        for (size_t i = 0; i < n; ++i) {
            Ct y = pg.unchecked_add(nl[i], pg.unchecked_scalar_mul(cr[i], 2));
            if (i + 1 < n) y = pg.unchecked_add(y, pg.unchecked_scalar_mul(nl[i + 1], 4));
            in_line[i] = pg.pbs(y, [](uint64_t x) { return uint64_t(!(x & 1) && (x & 6) != 6); });
            ends[i + 1] = nl[i];
        }
        const std::vector<Radix> cnt = prefix_count(nl, nd);
        const Ct trailing = isk.boolean_bitnot(end_part_empty(s, ends));
        const Radix count = isk.add(resized(cnt[n - 1], nd), resized({trailing}, nd));
        for (size_t k = 0; k < n; ++k) {
            std::vector<Ct> in(n, pg.create_trivial(0));
            for (size_t i = k; i < n; ++i) {                           // before char i there are at most i newlines
                const Radix before = i > 0 ? cnt[i - 1] : trivial_radix(0, nd);
                in[i] = pg.pbs_bivariate(scalar_sign(before, k), in_line[i], [](uint64_t sg, uint64_t l) {
                    return uint64_t(sg == IntegerServerKey::IS_EQUAL && (l & 1));
                });
            }
            if (k == 0) {   // line 0 starts at 0
                FheString p0;
                for (size_t i = 0; i < n; ++i) p0.chars.push_back(keep(s.chars[i], in[i]));
                parts.push_back(p0);
            } else parts.push_back(part(s, in));
        }
        return {count, parts};
    }

    // split_whitespace: the words between runs of char::is_whitespace, the 25 code points of Unicode White_Space: U+0009 ..= U+000D,
    // U+0020, U+0085, U+00A0, U+1680, U+2000 ..= U+200A, U+2028, U+2029, U+202F, U+205F, U+3000.  Every occurrence of their UTF-8
    // sequences is a separator: 09 ..= 0D, 20; C2 85, C2 A0; E1 9A 80, E2 80 80 ..= E2 80 8A, E2 80 A8, E2 80 A9, E2 80 AF, E2 81 9F,
    // E3 80 80.  For valid UTF-8 that is Rust's result (UTF-8 is self-synchronising); for other bytes this rule is the definition.  The
    // occurrences never overlap (each starts at an ASCII or lead byte, the rest are continuation bytes).
    // Each byte is classified once: two high-nibble and five low-nibble codes, then seven table lookups give its roles (separator byte or
    // padding, C2, lead E1 / E2 / E3, second byte 9A / 80 / 81, C2's second byte 85 / A0, third byte 80 / {81 ..= 8A, A8, A9, AF} / 9F);
    // neighbours are combined by three more lookups ("second and third byte", "lead and tail", "C2 and its second byte") and the word
    // flag is one lookup on the sum of the covering occurrences: 18 PBS per byte
    std::vector<Ct> unicode_word_chars(const FheString &s) {
        const size_t n = s.len();
        static uint64_t (*const hW)(uint64_t) = [](uint64_t h) { return h == 0 ? uint64_t(1) : h == 2 ? uint64_t(2) : h == 0xC ? uint64_t(3) : h == 0xE ? uint64_t(4) : uint64_t(0); };
        static uint64_t (*const hK)(uint64_t) = [](uint64_t h) { return h == 8 ? uint64_t(1) : h == 9 ? uint64_t(2) : h == 0xA ? uint64_t(3) : uint64_t(0); };
        static uint64_t (*const lW)(uint64_t) = [](uint64_t l) { return l == 0 ? uint64_t(1) : (l >= 9 && l <= 0xD) ? uint64_t(2) : uint64_t(0); };
        static uint64_t (*const lL)(uint64_t) = [](uint64_t l) { return l >= 1 && l <= 3 ? l : uint64_t(0); };
        static uint64_t (*const lA)(uint64_t) = [](uint64_t l) { return l == 0 ? uint64_t(1) : l == 1 ? uint64_t(2) : l == 0xA ? uint64_t(3) : uint64_t(0); };
        static uint64_t (*const lB)(uint64_t) = [](uint64_t l) { return (l >= 2 && l <= 7) ? uint64_t(1) : (l == 8 || l == 9) ? uint64_t(2) : l == 0xF ? uint64_t(3) : uint64_t(0); };
        static uint64_t (*const lE)(uint64_t) = [](uint64_t l) { return l == 0 ? uint64_t(1) : l == 5 ? uint64_t(2) : uint64_t(0); };
        std::vector<Ct> brk(n), lead(n), c2(n), sec(n), s2(n), thd(n);
        for (size_t i = 0; i < n; ++i) {
            const Ct hi = high_nibble(s.chars[i]), lo = low_nibble(s.chars[i]);
            const Ct hw = nibble_code(hi, hW), hk = nibble_code(hi, hK);
            const Ct lw = nibble_code(lo, lW), ll = nibble_code(lo, lL), la = nibble_code(lo, lA), lb = nibble_code(lo, lB), le = nibble_code(lo, lE);
            brk[i] = byte_lookup(hw, lw, 3, hW, lW, [](uint64_t b) { return uint64_t(b == 0 || (b >= 0x09 && b <= 0x0D) || b == 0x20); });
            lead[i] = byte_lookup(hw, ll, 3, hW, lL, [](uint64_t b) { return b >= 0xE1 && b <= 0xE3 ? b - 0xE0 : uint64_t(0); });
            c2[i] = byte_lookup(hw, ll, 3, hW, lL, [](uint64_t b) { return uint64_t(b == 0xC2); });
            sec[i] = byte_lookup(hk, la, 4, hK, lA, [](uint64_t b) { return b == 0x9A ? uint64_t(1) : b == 0x80 ? uint64_t(2) : b == 0x81 ? uint64_t(3) : uint64_t(0); });
            s2[i] = byte_lookup(hk, le, 3, hK, lE, [](uint64_t b) { return uint64_t(b == 0x85 || b == 0xA0); });
            // third byte: 1 = 80, 2 = 81 ..= 8A, A8, A9, AF, 3 = 9F; the two lookups see disjoint low nibbles, so their sum is the code
            const Ct ta = byte_lookup(hk, la, 4, hK, lA, [](uint64_t b) { return b == 0x80 ? uint64_t(1) : (b == 0x81 || b == 0x8A) ? uint64_t(2) : uint64_t(0); });
            const Ct tb = byte_lookup(hk, lb, 4, hK, lB, [](uint64_t b) {
                return (b >= 0x82 && b <= 0x89) || b == 0xA8 || b == 0xA9 || b == 0xAF ? uint64_t(2) : b == 0x9F ? uint64_t(3) : uint64_t(0);
            });
            thd[i] = add_disjoint(ta, tb, 3);
        }
        // tail[j]: bytes j, j + 1 are 9A 80 (1: after E1), 80 80 (2: after E2 or E3), 80 {81 ..= 8A, A8, A9, AF} or 81 9F (3: after E2)
        std::vector<Ct> tail(n, pg.create_trivial(0)), occ3(n, pg.create_trivial(0)), occ2(n, pg.create_trivial(0));
        for (size_t j = 0; j + 1 < n; ++j)
            tail[j] = pg.pbs_bivariate(sec[j], thd[j + 1], [](uint64_t a, uint64_t t) {
                return a == 1 && t == 1 ? uint64_t(1) : a == 2 && t == 1 ? uint64_t(2) : (a == 2 && t == 2) || (a == 3 && t == 3) ? uint64_t(3) : uint64_t(0);
            });
        for (size_t i = 0; i + 2 < n; ++i)
            occ3[i] = pg.pbs_bivariate(lead[i], tail[i + 1], [](uint64_t l, uint64_t t) { return uint64_t((l == 1 && t == 1) || (l == 2 && t >= 2) || (l == 3 && t == 2)); });
        for (size_t i = 0; i + 1 < n; ++i)
            occ2[i] = pg.pbs_bivariate(c2[i], s2[i + 1], [](uint64_t a, uint64_t b) { return uint64_t((a & 1) && (b & 1)); });
        std::vector<Ct> word(n);
        for (size_t i = 0; i < n; ++i) {
            Ct y = pg.unchecked_add(brk[i], pg.unchecked_add(occ2[i], occ3[i]));
            if (i >= 1) y = pg.unchecked_add(y, pg.unchecked_add(occ2[i - 1], occ3[i - 1]));
            if (i >= 2) y = pg.unchecked_add(y, occ3[i - 2]);
            word[i] = pg.pbs(y, [](uint64_t x) { return uint64_t(x == 0); });
        }
        return word;
    }
    std::pair<Radix, std::vector<FheString>> split_whitespace(const FheString &s) { return words(s, unicode_word_chars(s)); }

    Program &pg;
    IntegerServerKey isk;
    StringServerKey ssk;
    Params p;
};

}  // namespace tbh
