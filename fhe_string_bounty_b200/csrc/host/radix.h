// host/radix.h -- mirror of the integer radix methods that feed the string ops, recorded as level-batched
// programs (host/program.h).  Reference (tfhe/src/integer/server_key/):
//   unchecked_eq/ne_parallelized                 radix_parallel/comparison.rs:10-83
//   are_all_comparisons_block_true               radix_parallel/scalar_comparison.rs:147-198
//   is_at_least_one_comparisons_block_true       radix_parallel/scalar_comparison.rs:200-240
//   pack_block_chunk / pack_block_assign         radix_parallel/scalar_comparison.rs:104-139
//   unchecked_scalar_eq/ne_parallelized          radix_parallel/scalar_comparison.rs:254-458
//   Comparator (sign blocks, reduction tree, map_sign_result)   comparator.rs:52-133,193-279,389-464,957-971,1103-1126
//   scalar compare                               comparator.rs:226-238,474-502
//   boolean_bitand/bitor/bitnot                  radix/bitwise_op.rs:632-739
//   if_then_else / zero_out_if                   radix_parallel/cmux.rs:72-,211-250,281-
//   carry propagation (Hillis-Steele)            radix_parallel/add.rs:518-603,724-772 ; radix_parallel/mod.rs:88-156
// A radix ciphertext is a little-endian vector of blocks (integer/ciphertext/mod.rs:18-30, encryption.rs:46-83).
#pragma once
#include "program.h"

namespace tbh {

using Radix = std::vector<Ct>;   // little-endian blocks
using BooleanBlock = Ct;         // integer/ciphertext/boolean_value.rs:46

class IntegerServerKey {
  public:
    explicit IntegerServerKey(Program &prog) : pg(prog), p(prog.params()) {}

    // ---- boolean count-trees (scalar_comparison.rs:147-240) -------------------------------------------------
    // booleans summed per PBS: total_mod - 1.  With a message space of two values a sum of one boolean never shrinks the list.
    size_t count_tree_arity(size_t n_blocks) const {
        const size_t max_value = p.total_mod() - 1;
        if (n_blocks > 1 && max_value < 2) throw std::invalid_argument("boolean reduction: needs a message space of at least 3 values");
        return max_value;
    }
    Ct are_all_comparisons_block_true(std::vector<Ct> blocks) {
        if (blocks.empty()) return pg.create_trivial(1);
        const size_t max_value = count_tree_arity(blocks.size());
        while (blocks.size() > 1) {
            std::vector<Ct> next;
            for (size_t i = 0; i < blocks.size(); i += max_value) {
                const size_t len = std::min(max_value, blocks.size() - i);
                Ct sum = blocks[i];
                for (size_t j = 1; j < len; ++j) sum = pg.unchecked_add(sum, blocks[i + j]);
                next.push_back(pg.pbs(sum, [len](uint64_t x) { return uint64_t(x == len); }));
            }
            blocks.swap(next);
        }
        return blocks[0];
    }
    Ct is_at_least_one_comparisons_block_true(std::vector<Ct> blocks) {
        if (blocks.empty()) return pg.create_trivial(1);   // sic: scalar_comparison.rs:204-206
        const size_t max_value = count_tree_arity(blocks.size());
        while (blocks.size() > 1) {
            std::vector<Ct> next;
            for (size_t i = 0; i < blocks.size(); i += max_value) {
                const size_t len = std::min(max_value, blocks.size() - i);
                Ct sum = blocks[i];
                for (size_t j = 1; j < len; ++j) sum = pg.unchecked_add(sum, blocks[i + j]);
                next.push_back(pg.pbs(sum, [](uint64_t x) { return uint64_t(x != 0); }));
            }
            blocks.swap(next);
        }
        return blocks[0];
    }

    // ---- equality (comparison.rs:10-83) ---------------------------------------------------------------------------
    std::vector<Ct> block_equalities(const Radix &lhs, const Radix &rhs, bool want_ne = false) {
        if (lhs.size() != rhs.size()) throw std::invalid_argument("radix size mismatch");
        std::vector<Ct> out;
        for (size_t i = 0; i < lhs.size(); ++i)
            out.push_back(want_ne ? pg.pbs_bivariate(lhs[i], rhs[i], [](uint64_t x, uint64_t y) { return uint64_t(x != y); })
                                  : pg.pbs_bivariate(lhs[i], rhs[i], [](uint64_t x, uint64_t y) { return uint64_t(x == y); }));
        return out;
    }
    BooleanBlock unchecked_eq(const Radix &lhs, const Radix &rhs) {
        return are_all_comparisons_block_true(block_equalities(lhs, rhs));
    }
    BooleanBlock unchecked_ne(const Radix &lhs, const Radix &rhs) {
        std::vector<Ct> cmp = block_equalities(lhs, rhs, true);
        if (cmp.empty()) return pg.create_trivial(0);       // comparison.rs:76-82
        return is_at_least_one_comparisons_block_true(cmp);
    }

    // ---- packed equality: not a reference method, but built from the reference's own pieces -- pack two blocks into
    // msg*msg values (pack_block_chunk, scalar_comparison.rs:104-139), true LWE subtraction and a LUT on the difference
    // exactly like Comparator::compare_block_assign (comparator.rs:193-221), with f(x) = [x == 0]: for a negative
    // difference the padding bit makes the PBS return -f(16 - |d|) = 0.  One PBS per PAIR of blocks instead of one per
    // block; decrypted results identical to unchecked_eq, noise of the PBS input as in the reference's comparisons.
    std::vector<Ct> packed_block_equalities(const Radix &lhs, const Radix &rhs) {
        if (lhs.size() != rhs.size()) throw std::invalid_argument("radix size mismatch");
        std::vector<Ct> pl = pack_pairs(lhs), pr = pack_pairs(rhs), out;
        // the difference lies in (-total_mod, total_mod) only if both packed operands fit the message space (carry_mod >= msg_mod for
        // clean blocks); otherwise hi * msg_mod + lo wraps and distinct pairs compare equal: one PBS per block instead
        for (size_t i = 0; i < pl.size(); ++i)
            if (pl[i].degree >= p.total_mod() || pr[i].degree >= p.total_mod()) return block_equalities(lhs, rhs);
        for (size_t i = 0; i < pl.size(); ++i) {
            Ct d = pg.lwe_sub(pl[i], pr[i]);
            d.degree = p.total_mod() - 1;      // negative differences reach the padding bit on purpose (see above)
            out.push_back(pg.pbs(d, [](uint64_t x) { return uint64_t(x == 0); }));
        }
        return out;
    }
    BooleanBlock unchecked_eq_packed(const Radix &lhs, const Radix &rhs) {
        return are_all_comparisons_block_true(packed_block_equalities(lhs, rhs));
    }

    // ---- scalar equality (scalar_comparison.rs:254-458): pack pairs of blocks to msg*msg, one LUT per scalar nibble-pair
    std::vector<Ct> pack_pairs(const Radix &blocks) {
        std::vector<Ct> packed;
        for (size_t i = 0; i < blocks.size(); i += 2) {
            if (i + 1 < blocks.size()) packed.push_back(pg.unchecked_add(pg.unchecked_scalar_mul(blocks[i + 1], p.msg_mod), blocks[i]));
            else packed.push_back(blocks[i]);
        }
        return packed;
    }
    BooleanBlock unchecked_scalar_eq(const Radix &lhs, uint64_t scalar) {
        // value must fit, otherwise the result is trivially false (scalar_comparison.rs:383-398)
        const unsigned bits_per_block = log2u(p.msg_mod);
        if (lhs.size() * bits_per_block < 64 && (scalar >> (lhs.size() * bits_per_block)) != 0) return pg.create_trivial(0);
        std::vector<Ct> packed = pack_pairs(lhs);
        std::vector<Ct> cmp;
        const uint64_t pm = uint64_t(p.msg_mod) * p.msg_mod;
        for (size_t i = 0; i < packed.size(); ++i) {
            const bool pair = 2 * i + 1 < lhs.size();
            const uint64_t mod = pair ? pm : p.msg_mod;
            const uint64_t sv = scalar % mod;
            scalar /= mod;
            cmp.push_back(pg.pbs(packed[i], [sv](uint64_t x) { return uint64_t(x == sv); }));
        }
        return are_all_comparisons_block_true(cmp);
    }

    // ---- Comparator (comparator.rs) -------------------------------------------------------------------------------
    static constexpr uint64_t IS_INFERIOR = 0, IS_EQUAL = 1, IS_SUPERIOR = 2;

    // comparator.rs:193-221: lwe_sub, PBS(x != 0) (padding-bit trick gives -1 for lhs < rhs), + 1  => {0,1,2}
    Ct compare_block(const Ct &lhs, const Ct &rhs) {
        Ct d = pg.lwe_sub(lhs, rhs);
        d.degree = p.total_mod() - 1;
        Ct s = pg.pbs(d, [](uint64_t x) { return uint64_t(x != 0); });
        return pg.unchecked_scalar_add(s, 1);
    }
    // comparator.rs:226-238
    Ct scalar_compare_block(const Ct &lhs, uint64_t scalar) {
        Ct d = pg.plaintext_sub(lhs, scalar);
        Ct s = pg.pbs(d, [](uint64_t x) { return uint64_t(x != 0); });
        return pg.unchecked_scalar_add(s, 1);
    }
    // comparator.rs:240-279: pairwise tree, high*4 + low through comparison_reduction_lut (:72-95)
    Ct reduce_signs(std::vector<Ct> signs) {
        auto reduction = [](uint64_t x) -> uint64_t {
            static const uint64_t t[11] = {0, 0, 0, 0, 0, 1, 2, 2, 2, 2, 2};
            return x < 11 ? t[x] : 0;
        };
        while (signs.size() != 1) {
            std::vector<Ct> next;
            for (size_t i = 0; i + 1 < signs.size(); i += 2) {
                Ct packed = pg.unchecked_add(pg.unchecked_scalar_mul(signs[i + 1], 4), signs[i]);
                next.push_back(pg.pbs(packed, reduction));
            }
            if (signs.size() % 2 == 1) next.push_back(signs.back());
            signs.swap(next);
        }
        return signs[0];
    }
    // comparator.rs:389-464 (unsigned; carry_modulus >= message_modulus branch: blocks packed two by two)
    Ct unchecked_compare(const Radix &lhs, const Radix &rhs) {
        if (lhs.size() != rhs.size() || lhs.empty()) throw std::invalid_argument("compare: radix size mismatch / empty");
        std::vector<Ct> cmp;
        if (p.carry_mod < p.msg_mod) {
            for (size_t i = 0; i < lhs.size(); ++i) cmp.push_back(compare_block(lhs[i], rhs[i]));
        } else {
            std::vector<Ct> pl = pack_pairs(lhs), pr = pack_pairs(rhs);
            for (size_t i = 0; i < pl.size(); ++i) cmp.push_back(compare_block(pl[i], pr[i]));
        }
        return reduce_signs(cmp);
    }
    // comparator.rs:474-502 (scalar on the right, packed blocks)
    Ct unchecked_scalar_compare(const Radix &lhs, uint64_t scalar) {
        if (lhs.empty()) throw std::invalid_argument("compare: empty radix");
        std::vector<Ct> packed = pack_pairs(lhs);
        const uint64_t pm = uint64_t(p.msg_mod) * p.msg_mod;
        std::vector<Ct> cmp;
        for (size_t i = 0; i < packed.size(); ++i) {
            const bool pair = 2 * i + 1 < lhs.size();
            const uint64_t mod = pair ? pm : p.msg_mod;
            cmp.push_back(scalar_compare_block(packed[i], scalar % mod));
            scalar /= mod;
        }
        Ct sign = reduce_signs(cmp);
        if (scalar != 0)  // scalar has bits above the radix: lhs < scalar regardless (comparator.rs:677-)
            return pg.unchecked_create_trivial(IS_INFERIOR);
        return sign;
    }
    // comparator.rs:957-971
    BooleanBlock map_sign_result(const Ct &sign, const std::function<bool(uint64_t)> &h) {
        return pg.pbs(sign, [h](uint64_t x) { return uint64_t(h(x)); });
    }
    BooleanBlock unchecked_lt(const Radix &a, const Radix &b) { return map_sign_result(unchecked_compare(a, b), [](uint64_t x) { return x == IS_INFERIOR; }); }
    BooleanBlock unchecked_le(const Radix &a, const Radix &b) { return map_sign_result(unchecked_compare(a, b), [](uint64_t x) { return x == IS_INFERIOR || x == IS_EQUAL; }); }
    BooleanBlock unchecked_gt(const Radix &a, const Radix &b) { return map_sign_result(unchecked_compare(a, b), [](uint64_t x) { return x == IS_SUPERIOR; }); }
    BooleanBlock unchecked_ge(const Radix &a, const Radix &b) { return map_sign_result(unchecked_compare(a, b), [](uint64_t x) { return x == IS_SUPERIOR || x == IS_EQUAL; }); }
    BooleanBlock unchecked_scalar_lt(const Radix &a, uint64_t s) { return map_sign_result(unchecked_scalar_compare(a, s), [](uint64_t x) { return x == IS_INFERIOR; }); }
    BooleanBlock unchecked_scalar_gt(const Radix &a, uint64_t s) { return map_sign_result(unchecked_scalar_compare(a, s), [](uint64_t x) { return x == IS_SUPERIOR; }); }

    // ---- booleans (radix/bitwise_op.rs:632-739) -------------------------------------------------------------------------
    BooleanBlock boolean_bitand(const Ct &a, const Ct &b) { return pg.pbs_bivariate(a, b, [](uint64_t x, uint64_t y) { return (x & y) & 1; }); }
    BooleanBlock boolean_bitor(const Ct &a, const Ct &b) { return pg.pbs_bivariate(a, b, [](uint64_t x, uint64_t y) { return (x | y) & 1; }); }
    // scalar xor 1 on a clean boolean == 1 - x: leveled (bitwise_op.rs:720-739 uses scalar_bitxor; same decrypted value)
    BooleanBlock boolean_bitnot(const Ct &a) {
        Ct r = pg.unchecked_scalar_add(pg.unchecked_scalar_mul(a, uint64_t(-1)), 1);
        r.degree = 1; r.noise = a.noise;
        return r;
    }

    // ---- cmux (radix_parallel/cmux.rs:211-250): result_i = cond ? a_i : b_i -------------------------------------------------
    Radix if_then_else(const Ct &cond, const Radix &a, const Radix &b) {
        if (a.size() != b.size()) throw std::invalid_argument("cmux: radix size mismatch");
        Radix out;
        for (size_t i = 0; i < a.size(); ++i) {
            // zero_out_if (cmux.rs:281-): block * msg_mod + cond through a bivariate LUT
            Ct ta = pg.pbs_bivariate(a[i], cond, [](uint64_t blk, uint64_t c) { return c ? blk : uint64_t(0); });
            Ct tb = pg.pbs_bivariate(b[i], cond, [](uint64_t blk, uint64_t c) { return c ? uint64_t(0) : blk; });
            Ct sum = pg.unchecked_add(ta, tb);                       // exactly one of the two is non-zero
            out.push_back(pg.pbs(sum, [this](uint64_t x) { return x % p.msg_mod; }));   // message_extract
        }
        return out;
    }

    // ---- carry propagation (radix_parallel/add.rs:518-603,724-772), always the parallel form (SURVEY App. B note) ---------------
    // blocks hold message + at most one carry (degree <= 2 msg_mod - 2, so that block + incoming carry <= 2 msg_mod - 1 carries out at
    // most one); returns clean blocks of the propagated number (mod msg_mod^B)
    Radix full_propagate(const Radix &in) {
        const uint64_t m = p.msg_mod;
        const size_t B = in.size();
        if (B == 0) return in;
        for (auto &b : in)
            if (b.degree > 2 * m - 2) throw std::logic_error("single-carry propagation on a block of degree " + std::to_string(b.degree));
        enum : uint64_t { NONE = 0, GENERATED = 1, PROPAGATED = 2 };   // add.rs:19-34 OutputCarry
        // generate_init_carry_array (add.rs:724-772): first block can only generate
        std::vector<Ct> state(B);
        for (size_t i = 0; i < B; ++i) {
            if (i == 0) state[i] = pg.pbs(in[i], [m](uint64_t x) { return uint64_t(x >= m ? GENERATED : NONE); });
            else state[i] = pg.pbs(in[i], [m](uint64_t x) { return x >= m ? uint64_t(GENERATED) : (x == m - 1 ? uint64_t(PROPAGATED) : uint64_t(NONE)); });
        }
        // Hillis-Steele inclusive prefix (add.rs:572-603) with prefix_sum_carry_propagation (add.rs:36-42)
        // the pair (cur, prev) of states in {0, 1, 2} is packed as cur * msg_mod + prev; with msg_mod = 2 that is not injective, so the
        // one-bit sets pack it as cur * 3 + prev (a univariate LUT on [0, 8]: a message space of at least 9 values)
        auto combine = [](uint64_t cur, uint64_t prev) { return cur == PROPAGATED ? prev : cur; };
        for (size_t d = 1; d < B; d *= 2) {
            std::vector<Ct> next = state;
            for (size_t i = d; i < B; ++i) {
                if (m >= 3) next[i] = pg.pbs_bivariate(state[i], state[i - d], combine);
                else next[i] = pg.pbs(pg.unchecked_add(pg.unchecked_scalar_mul(state[i], 3), state[i - d]),
                                      [combine](uint64_t x) { return x < 9 ? combine(x / 3, x % 3) : uint64_t(0); });
            }
            state.swap(next);
        }
        // add the incoming carry and extract the message (add.rs:544-570)
        Radix out(B);
        for (size_t i = 0; i < B; ++i) {
            Ct v = in[i];
            // after the full inclusive prefix every state is NONE (0) or GENERATED (1) -- block 0 can never be
            // PROPAGATED -- so the state IS the carry bit (add.rs:544-570: unchecked_add_assign(block, carry))
            if (i > 0) v = pg.unchecked_add(v, state[i - 1]);
            out[i] = pg.pbs(v, [m](uint64_t x) { return x % m; });
        }
        return out;
    }
    // full_propagate_parallelized on blocks of ANY degree < total_mod (radix_parallel/mod.rs:88-156, parallel branch): message_extract
    // and carry_extract of every block in one level, the carries added one block up, then the single-carry propagation above.  One
    // extraction leaves message + carry <= (msg_mod - 1) + (d / msg_mod); when carry_mod > msg_mod that can still exceed 2 msg_mod - 2,
    // so the extraction repeats until every block allows a single carry.  Blocks that already do go straight to it.
    Radix full_propagate_any_degree(Radix in) {
        const uint64_t m = p.msg_mod;
        auto worst_of = [](const Radix &r) { uint64_t w = 0; for (auto &b : r) w = std::max(w, b.degree); return w; };
        while (worst_of(in) > 2 * m - 2) {
            Radix msg(in.size()), carry(in.size());
            for (size_t i = 0; i < in.size(); ++i) {
                msg[i] = pg.pbs(in[i], [m](uint64_t x) { return x % m; });
                msg[i].degree = std::min(in[i].degree, m - 1);
                if (i + 1 < in.size()) {
                    carry[i] = pg.pbs(in[i], [m](uint64_t x) { return x / m; });
                    carry[i].degree = in[i].degree / m;
                }
            }
            for (size_t i = 1; i < in.size(); ++i) msg[i] = pg.unchecked_add(msg[i], carry[i - 1]);
            in.swap(msg);
        }
        return full_propagate(in);
    }
    bool block_carries_are_empty(const Radix &r) const {      // integer/ciphertext/base.rs: every degree < msg_mod
        for (auto &b : r) if (b.degree >= p.msg_mod) return false;
        return true;
    }
    // the default (non-"unchecked") comparisons: propagate an operand first if its carries are not empty (comparison.rs:200-260)
    Radix cleaned(const Radix &r) { return block_carries_are_empty(r) ? r : full_propagate_any_degree(r); }

    // add_parallelized on clean inputs (radix_parallel/add.rs:206-243): leveled add then propagate
    Radix add(const Radix &a, const Radix &b) {
        if (a.size() != b.size()) throw std::invalid_argument("add: radix size mismatch");
        Radix s(a.size());
        for (size_t i = 0; i < a.size(); ++i) s[i] = pg.unchecked_add(a[i], b[i]);
        return full_propagate(s);
    }

    static unsigned log2u(uint64_t x) { unsigned l = 0; while ((uint64_t(1) << l) < x) ++l; return l; }

    Program &pg;
    Params p;
};

}  // namespace tbh
