// host_api.cu -- C ABI of the host layer: record an integer / string operation as a level-batched program
// (host/program.h, host/radix.h, host/strings.h), inspect it without a GPU, and execute it on a context:
// per level ONE leveled-op launch + ONE keyswitch launch + ONE PBS launch over every independent block.
// This is the restructuring of the reference's per-block rayon fan-out
// (integer/server_key/radix_parallel/*.rs -> shortint apply_lookup_table) that north_star asks for.
#include "ctx.h"
#include "host/padded.h"
#include "../../include/tfhe_b200_sharded.h"

#include <cstring>
#include <deque>
#include <memory>

using tbc::DevBuf;
using tbc::DeviceGuard;
using tbc::fail;

struct tfhe_b200_program {
    tbh::Params p;
    std::unique_ptr<tbh::LutRegistry> luts;
    std::unique_ptr<tbh::Program> prog;
    std::string op;
    // device copies, valid for the context with id `owner_id` on CUDA device `device` (ids are unique per process, so a destroyed
    // context whose address is reused is never mistaken for the owner; the buffers are plain device memory and outlive the context)
    uint64_t owner_id = 0;
    int device = -1;
    DevBuf d_luts, d_lin, d_terms, d_pbs_in, d_pbs_out, d_pbs_lut, d_arena, d_out_slots, d_out_rows;
    std::vector<uint32_t> lin_off, pbs_off;   // per level offsets
    float last_ms = 0.f;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // recorded after the last launch of a run that reads d_arena (the output gather): a run on any stream waits for it before it writes
    // its inputs there (tbc::StreamOrder)
    cudaEvent_t arena_done = nullptr;
};

namespace {

tbh::Params to_host_params(const tfhe_b200_params &q) {
    return tbh::Params{q.lwe_dim, q.glwe_dim, q.poly_size, q.pbs_base_log, q.pbs_level, q.ks_base_log, q.ks_level,
                       q.grouping_factor, q.msg_mod, q.carry_mod};
}

tbh::Radix input_radix(tbh::Program &pg, size_t n) {
    tbh::Radix r;
    for (size_t i = 0; i < n; ++i) r.push_back(pg.input());
    return r;
}

void output_radix(tbh::Program &pg, const tbh::Radix &r) { for (auto &b : r) pg.output(b); }
void output_string(tbh::Program &pg, const tbh::FheString &s) { for (auto &c : s.chars) output_radix(pg, c); }

// pstring_{replace,replacen} {capacity, capacity_from, capacity_to[, count]}: inputs s, from, to -> the result string
// pstring_{split,splitn} {capacity, capacity_pat[, n]}: inputs s, pat -> part count, then the parts
// pstring_{split_once,rsplit_once} {capacity, capacity_pat}: inputs s, pat -> found, before, after
// A clear pattern replaces the `from` / `pat` input; its capacity argument must be its length.
bool record_split_replace(tbh::Program &pg, tbh::PaddedStringServerKey &psk, tbh::StringServerKey &ssk, const std::string &op,
                          const std::string &f, const uint64_t *a, size_t na, const char *clear, std::string &err) {
    const bool rep = f == "replace" || f == "replacen";
    const size_t n_args = f == "replacen" ? 4 : (f == "replace" || f == "splitn") ? 3 : 2;
    if (na < n_args) {
        static const std::map<std::string, std::string> names = {
            {"replace", "{capacity, capacity_from, capacity_to}"}, {"replacen", "{capacity, capacity_from, capacity_to, count}"},
            {"split", "{capacity, capacity_pat}"}, {"splitn", "{capacity, capacity_pat, n}"},
            {"split_once", "{capacity, capacity_pat}"}, {"rsplit_once", "{capacity, capacity_pat}"}};
        err = op + ": expected " + std::to_string(n_args) + " integer arguments " + names.at(f);
        return false;
    }
    const uint64_t cap = a[0], cap_pat = a[1], cap_to = rep ? a[2] : 0;
    if (clear && std::strlen(clear) != cap_pat) {
        err = op + ": the pattern capacity " + std::to_string(cap_pat) + " differs from the clear pattern's length " + std::to_string(std::strlen(clear));
        return false;
    }
    // sizes arrive from outside: bound the result and the intermediate strings before anything is recorded (slot indices are 32-bit)
    constexpr uint64_t kMaxChars = uint64_t(1) << 20;
    if (cap > kMaxChars || cap_pat > kMaxChars || cap_to > kMaxChars) {
        err = op + ": capacities are limited to " + std::to_string(kMaxChars) + " chars";
        return false;
    }
    const uint64_t m_min = clear ? cap_pat : 0, M = tbh::PaddedStringServerKey::max_matches(cap, m_min);
    unsigned __int128 chars;   // the largest string the program holds at once
    if (rep) {
        const uint64_t count = f == "replacen" ? std::min<uint64_t>(a[3], M) : M;
        chars = (unsigned __int128)(cap + 1) * (cap_to + 1);                                        // the expanded string
        chars = std::max(chars, (unsigned __int128)cap + (unsigned __int128)count * (cap_to > m_min ? cap_to - m_min : 0));
    } else {
        const uint64_t P = f == "splitn" ? std::min<uint64_t>(M + 1, a[2]) : (f == "split" ? M + 1 : 2);
        chars = (unsigned __int128)P * cap;
    }
    if (chars > kMaxChars) {
        err = op + ": the result or the expanded string would exceed " + std::to_string(kMaxChars) + " chars";
        return false;
    }
    tbh::FheString s = ssk.input_string(cap);
    const tbh::PaddedStringServerKey::Pattern pt = clear ? psk.clear_pattern(clear) : psk.padded_pattern(ssk.input_string(cap_pat));
    if (rep) {
        tbh::FheString to = ssk.input_string(cap_to);
        output_string(pg, psk.replace(s, pt, to, f == "replacen" ? a[3] : SIZE_MAX));
    } else if (f == "split" || f == "splitn") {
        auto r = psk.split(s, pt, f == "splitn" ? a[2] : SIZE_MAX);
        output_radix(pg, r.first);
        for (auto &part : r.second) output_string(pg, part);
    } else {
        auto r = psk.split_once(s, pt, f == "rsplit_once");
        pg.output(std::get<0>(r));
        output_string(pg, std::get<1>(r));
        output_string(pg, std::get<2>(r));
    }
    return true;
}

// The rest of the split family, the ops with a secret integer argument, the padded-pattern strip_prefix / strip_suffix, the padded
// eq_ignore_case, matches / match_indices / rmatch_indices / trim_start_matches / trim_end_matches, lines and split_whitespace;
// include/tfhe_b200.h gives every output layout.  A secret integer is a radix input of count_blocks blocks appended after
// the strings.  Every argument is checked before anything is recorded.
bool record_padded_extra(tbh::Program &pg, tbh::PaddedStringServerKey &psk, tbh::StringServerKey &ssk, const std::string &op,
                         const std::string &f, const uint64_t *a, size_t na, const char *clear, std::string &err) {
    static const std::map<std::string, std::vector<std::string>> kArgs = {
        {"rsplit", {"capacity", "capacity_pat"}}, {"rsplitn", {"capacity", "capacity_pat", "n"}},
        {"split_terminator", {"capacity", "capacity_pat"}}, {"rsplit_terminator", {"capacity", "capacity_pat"}},
        {"split_inclusive", {"capacity", "capacity_pat"}}, {"split_ascii_whitespace", {"capacity"}},
        {"repeat_enc", {"capacity", "max_count", "count_blocks"}},
        {"replacen_enc", {"capacity", "capacity_from", "capacity_to", "count_blocks"}},
        {"splitn_enc", {"capacity", "capacity_pat", "n_blocks"}}, {"rsplitn_enc", {"capacity", "capacity_pat", "n_blocks"}},
        {"strip_prefix", {"capacity", "capacity_pat"}}, {"strip_suffix", {"capacity", "capacity_pat"}},
        {"eq_ignore_case", {"capacity_a", "capacity_b"}},
        {"matches", {"capacity", "capacity_pat"}}, {"match_indices", {"capacity", "capacity_pat"}},
        {"rmatch_indices", {"capacity", "capacity_pat"}}, {"trim_start_matches", {"capacity", "capacity_pat"}},
        {"trim_end_matches", {"capacity", "capacity_pat"}}, {"lines", {"capacity"}}, {"split_whitespace", {"capacity"}}};
    const std::vector<std::string> &names = kArgs.at(f);
    if (na < names.size()) {
        std::string list;
        for (auto &nm : names) list += (list.empty() ? "" : ", ") + nm;
        err = op + ": expected " + std::to_string(names.size()) + " integer arguments {" + list + "}";
        return false;
    }
    const bool has_pattern = names.size() > 1 && names[1] != "max_count";
    if (clear && !has_pattern) {
        err = op + ": takes no clear operand";
        return false;
    }
    if (clear && std::strlen(clear) != a[1]) {
        err = op + ": the pattern capacity " + std::to_string(a[1]) + " differs from the clear pattern's length " + std::to_string(std::strlen(clear));
        return false;
    }
    const bool secret = f.size() > 4 && f.compare(f.size() - 4, 4, "_enc") == 0;
    const uint64_t blocks = secret ? a[names.size() - 1] : 0;
    if (secret && (blocks < 1 || blocks > 16)) {
        err = op + ": " + names.back() + " must be 1 ..= 16, got " + std::to_string(blocks);
        return false;
    }
    // sizes arrive from outside: bound every string and the result before anything is recorded (slot indices are 32-bit)
    constexpr uint64_t kMaxChars = uint64_t(1) << 20;
    const size_t n_sizes = names.size() - (secret || f == "rsplitn" ? 1 : 0);   // capacities (and repeat_enc's max_count)
    for (size_t i = 0; i < n_sizes; ++i)
        if (a[i] > kMaxChars) {
            err = op + ": capacities are limited to " + std::to_string(kMaxChars) + " chars";
            return false;
        }
    const uint64_t cap = a[0], m_min = clear ? a[1] : 0, M = tbh::PaddedStringServerKey::max_matches(cap, m_min);
    unsigned __int128 chars = cap;   // the largest string the program holds at once
    if (f == "repeat_enc") chars = (unsigned __int128)cap * a[1];
    else if (f == "replacen_enc") {
        const uint64_t cap_to = a[2];
        chars = std::max((unsigned __int128)(cap + 1) * (cap_to + 1), (unsigned __int128)cap + (unsigned __int128)M * (cap_to > m_min ? cap_to - m_min : 0));
    } else if (f == "split_ascii_whitespace" || f == "split_whitespace") chars = (unsigned __int128)((cap + 1) / 2) * cap;
    else if (f == "lines") chars = (unsigned __int128)cap * cap;
    else if (f == "match_indices" || f == "rmatch_indices") chars = (unsigned __int128)M * (cap + 1);   // one selection flag per match and window
    else if (f.find("split") != std::string::npos) chars = (unsigned __int128)(f == "rsplitn" ? std::min<uint64_t>(M + 1, a[2]) : M + 1) * cap;
    if (chars > kMaxChars) {
        err = op + ": the result or the expanded string would exceed " + std::to_string(kMaxChars) + " chars";
        return false;
    }

    tbh::FheString s = ssk.input_string(cap);
    if (f == "split_ascii_whitespace" || f == "split_whitespace" || f == "lines") {
        auto r = f == "lines" ? psk.lines(s) : f == "split_whitespace" ? psk.split_whitespace(s) : psk.split_ascii_whitespace(s);
        output_radix(pg, r.first);
        for (auto &part : r.second) output_string(pg, part);
        return true;
    }
    if (f == "repeat_enc") {
        tbh::Radix count = input_radix(pg, blocks);
        output_string(pg, psk.repeat(s, count, a[1]));
        return true;
    }
    if (f == "eq_ignore_case") {
        tbh::FheString t = clear ? ssk.trivial_string(clear) : ssk.input_string(a[1]);
        pg.output(psk.eq_ignore_case(s, t));
        return true;
    }
    if (f == "strip_prefix" || f == "strip_suffix") {   // the padded pattern (a clear one takes the form without capacity_pat)
        tbh::FheString pat = ssk.input_string(a[1]);
        auto r = f == "strip_prefix" ? psk.strip_prefix(s, pat) : psk.strip_suffix(s, pat);
        pg.output(r.first);
        output_string(pg, r.second);
        return true;
    }
    const tbh::PaddedStringServerKey::Pattern pt = clear ? psk.clear_pattern(clear) : psk.padded_pattern(ssk.input_string(a[1]));
    if (f == "replacen_enc") {
        tbh::FheString to = ssk.input_string(a[2]);
        tbh::Radix count = input_radix(pg, blocks);
        output_string(pg, psk.replace(s, pt, to, SIZE_MAX, &count));
        return true;
    }
    if (f == "matches") {
        output_radix(pg, psk.matches(s, pt));
        return true;
    }
    if (f == "match_indices" || f == "rmatch_indices") {
        auto r = psk.match_indices(s, pt, f == "rmatch_indices");
        output_radix(pg, r.first);
        for (auto &idx : r.second) output_radix(pg, idx);
        return true;
    }
    if (f == "trim_start_matches" || f == "trim_end_matches") {
        output_string(pg, f == "trim_start_matches" ? psk.trim_start_matches(s, pt) : psk.trim_end_matches(s, pt));
        return true;
    }
    std::pair<tbh::Radix, std::vector<tbh::FheString>> r;
    const bool reverse = f[0] == 'r';
    if (f == "split_inclusive") r = psk.split_inclusive(s, pt);
    else if (secret) {
        tbh::Radix n = input_radix(pg, blocks);
        r = psk.split(s, pt, SIZE_MAX, reverse, false, &n);
    } else r = psk.split(s, pt, f == "rsplitn" ? a[2] : SIZE_MAX, reverse, f.find("terminator") != std::string::npos);
    output_radix(pg, r.first);
    for (auto &part : r.second) output_string(pg, part);
    return true;
}

// records `op`; returns false with a message when the op / arguments are unknown
bool record(tfhe_b200_program &h, const std::string &op_in, const uint64_t *a, size_t na, const char *clear, std::string &err) {
    tbh::Program &pg = *h.prog;
    tbh::IntegerServerKey isk(pg);
    // "<op>_packed": same operation with packed block equalities (one PBS per pair of blocks, host/radix.h)
    std::string op = op_in;
    bool packed = false;
    if (op.size() > 7 && op.compare(op.size() - 7, 7, "_packed") == 0) { packed = true; op = op.substr(0, op.size() - 7); }
    tbh::StringServerKey ssk(pg, packed);
    if (packed && op == "radix_eq") {
        if (na < 1) { err = "radix_eq_packed: expected 1 integer argument"; return false; }
        tbh::Radix x = input_radix(pg, a[0]), y = input_radix(pg, a[0]);
        pg.output(isk.unchecked_eq_packed(x, y));
        return true;
    }
    auto need = [&](size_t n) { if (na < n) { err = op + ": expected " + std::to_string(n) + " integer arguments"; return false; } return true; };
    const std::string cl = clear ? clear : "";

    // ---- shortint level: one apply_lookup_table per input, LUT given as a table in `a` --------------------------------------
    if (op == "shortint_apply_lut") {            // a = {n_cts, f(0), ..., f(total_mod-1)}
        if (!need(1 + h.p.total_mod())) return false;
        std::vector<uint64_t> t(a + 1, a + 1 + h.p.total_mod());
        std::vector<tbh::Ct> in;
        for (size_t i = 0; i < a[0]; ++i) in.push_back(pg.input(h.p.total_mod() - 1, 1));
        for (auto &c : in) pg.output(pg.pbs(c, [t](uint64_t x) { return t[x]; }));
        return true;
    }
    if (op == "shortint_bivariate_lut") {        // a = {n_pairs, f(0,0), f(0,1), ..., f(m-1,m-1)}  row-major in (lhs, rhs)
        const size_t m = h.p.msg_mod;
        if (!need(1 + m * m)) return false;
        std::vector<uint64_t> t(a + 1, a + 1 + m * m);
        std::vector<tbh::Ct> l, r;
        for (size_t i = 0; i < a[0]; ++i) l.push_back(pg.input());
        for (size_t i = 0; i < a[0]; ++i) r.push_back(pg.input());
        for (size_t i = 0; i < a[0]; ++i) pg.output(pg.pbs_bivariate(l[i], r[i], [t, m](uint64_t x, uint64_t y) { return t[x * m + y]; }));
        return true;
    }
    // ---- integer radix level: a = {n_blocks[, scalar]} ---------------------------------------------------------------------------------
    if (op.rfind("radix_", 0) == 0) {
        if (!need(1)) return false;
        const size_t nb = a[0];
        const std::string f = op.substr(6);
        if (f == "scalar_eq" || f == "scalar_lt" || f == "scalar_gt") {
            if (!need(2)) return false;
            tbh::Radix x = input_radix(pg, nb);
            pg.output(f == "scalar_eq" ? isk.unchecked_scalar_eq(x, a[1]) : f == "scalar_lt" ? isk.unchecked_scalar_lt(x, a[1]) : isk.unchecked_scalar_gt(x, a[1]));
            return true;
        }
        // default (propagating) forms on operands whose blocks carry up to a[1] (e.g. 6 after one unchecked_add): what the reference's
        // comparison tests exercise (radix_parallel/tests_cases_comparisons.rs:81-97)
        if (f.rfind("default_", 0) == 0 || f == "full_propagate") {
            if (!need(2)) return false;
            if (a[1] >= h.p.total_mod()) { err = op + ": block degree must stay below the message space"; return false; }
            auto dirty = [&](size_t n) { tbh::Radix r; for (size_t i = 0; i < n; ++i) r.push_back(pg.input(a[1], 2)); return r; };
            tbh::Radix x = dirty(nb);
            if (f == "full_propagate") { output_radix(pg, isk.full_propagate_any_degree(x)); return true; }
            tbh::Radix y = dirty(nb);
            x = isk.cleaned(x); y = isk.cleaned(y);
            const std::string g = f.substr(8);
            if (g == "eq") pg.output(isk.unchecked_eq(x, y));
            else if (g == "ne") pg.output(isk.unchecked_ne(x, y));
            else if (g == "lt") pg.output(isk.unchecked_lt(x, y));
            else if (g == "le") pg.output(isk.unchecked_le(x, y));
            else if (g == "gt") pg.output(isk.unchecked_gt(x, y));
            else if (g == "ge") pg.output(isk.unchecked_ge(x, y));
            else { err = "unknown radix op: " + op; return false; }
            return true;
        }
        if (f == "if_then_else") {
            tbh::Ct cond = pg.input(1, 1);
            tbh::Radix x = input_radix(pg, nb), y = input_radix(pg, nb);
            output_radix(pg, isk.if_then_else(cond, x, y));
            return true;
        }
        tbh::Radix x = input_radix(pg, nb), y = input_radix(pg, nb);
        if (f == "eq") pg.output(isk.unchecked_eq(x, y));
        else if (f == "ne") pg.output(isk.unchecked_ne(x, y));
        else if (f == "lt") pg.output(isk.unchecked_lt(x, y));
        else if (f == "le") pg.output(isk.unchecked_le(x, y));
        else if (f == "gt") pg.output(isk.unchecked_gt(x, y));
        else if (f == "ge") pg.output(isk.unchecked_ge(x, y));
        else if (f == "add") output_radix(pg, isk.add(x, y));
        else { err = "unknown radix op: " + op; return false; }
        return true;
    }
    // ---- boolean reductions used by the multi-GPU split: a = {n_blocks}; inputs are boolean blocks -------------------------------------------
    if (op == "bool_all_true" || op == "bool_any_true") {
        if (!need(1)) return false;
        std::vector<tbh::Ct> b;
        for (size_t i = 0; i < a[0]; ++i) b.push_back(pg.input(1, 1));
        pg.output(op == "bool_all_true" ? isk.are_all_comparisons_block_true(b) : isk.is_at_least_one_comparisons_block_true(b));
        return true;
    }
    // final LUT after an all-reduce(SUM) of per-GPU boolean blocks: a = {n_summed, want_all}
    if (op == "bool_sum_finish") {
        if (!need(2)) return false;
        const uint64_t n = a[0];
        tbh::Ct s = pg.input(n, n);
        pg.output(a[1] ? pg.pbs(s, [n](uint64_t x) { return uint64_t(x == n); }) : pg.pbs(s, [](uint64_t x) { return uint64_t(x != 0); }));
        return true;
    }
    // ---- multi-GPU finishing programs (SURVEY 8e): inputs are what the ranks exchanged -------------------------------------------------
    if (op == "signs_finish") {                  // a = {count, want_less, or_equal}; inputs: count sign blocks, least significant range first
        if (!need(3)) return false;
        if (a[0] < 1) { err = "signs_finish: needs at least one sign block"; return false; }
        std::vector<tbh::Ct> signs;
        for (uint64_t r = 0; r < a[0]; ++r) signs.push_back(pg.input(2, 1));
        pg.output(ssk.finish_signs(signs, a[1] != 0, a[2] != 0));
        return true;
    }
    if (op == "find_combine") {                  // a = {count, index blocks}; inputs: count x (found flag, index radix), ascending window ranges
        if (!need(2)) return false;
        if (a[0] < 1 || 2 * a[0] > h.p.total_mod() || a[1] < 1) { err = "find_combine: 1..total_mod/2 parts, at least one index block"; return false; }
        std::vector<std::pair<tbh::Ct, tbh::Radix>> parts;
        for (uint64_t r = 0; r < a[0]; ++r) {
            tbh::Ct f = pg.input(1, 1);
            tbh::Radix idx;
            for (uint64_t b = 0; b < a[1]; ++b) idx.push_back(pg.input(h.p.msg_mod - 1, 1));
            parts.push_back({f, idx});
        }
        auto r = ssk.combine_find(parts);
        pg.output(r.first);
        output_radix(pg, r.second);
        return true;
    }
    // ---- many independent string pairs in one program (throughput mode): a = {len_a, len_b, count}; inputs are
    //      count x (string a, string b); one boolean per pair.  op = string_eq_many / string_lt_many / string_contains_many
    if (op.size() > 5 && op.rfind("string_", 0) == 0 && op.compare(op.size() - 5, 5, "_many") == 0) {
        if (!need(3)) return false;
        const std::string f = op.substr(7, op.size() - 12);
        std::vector<std::pair<tbh::FheString, tbh::FheString>> in;
        for (uint64_t k = 0; k < a[2]; ++k) {
            tbh::FheString s = ssk.input_string(a[0]);
            tbh::FheString t = ssk.input_string(a[1]);
            in.push_back({s, t});
        }
        for (auto &st : in) {
            if (f == "eq") pg.output(ssk.eq(st.first, st.second));
            else if (f == "ne") pg.output(ssk.ne(st.first, st.second));
            else if (f == "lt") pg.output(ssk.lt(st.first, st.second));
            else if (f == "le") pg.output(ssk.le(st.first, st.second));
            else if (f == "contains") pg.output(ssk.contains(st.first, st.second));
            else { err = "unknown batched string op: " + op; return false; }
        }
        return true;
    }
    // ---- null-padded strings (secret length, host/padded.h): a = {capacity_a[, capacity_b | count]}; a clear pattern comes through `clear` -----
    if (op.rfind("pstring_", 0) == 0) {
        if (!need(1)) return false;
        tbh::PaddedStringServerKey psk(pg);
        const std::string f = op.substr(8);
        if (f == "replace" || f == "replacen" || f == "split" || f == "splitn" || f == "split_once" || f == "rsplit_once")
            return record_split_replace(pg, psk, ssk, op, f, a, na, clear, err);
        if (f == "strip_prefix" || f == "strip_suffix") {
            if (!clear && na < 2) { err = op + ": needs a clear pattern, or {capacity, capacity_pat} and a padded pattern input"; return false; }
            if (!clear) return record_padded_extra(pg, psk, ssk, op, f, a, na, clear, err);
        }
        if (f == "rsplit" || f == "rsplitn" || f == "split_terminator" || f == "rsplit_terminator" || f == "split_inclusive" ||
            f == "split_ascii_whitespace" || f == "repeat_enc" || f == "replacen_enc" || f == "splitn_enc" || f == "rsplitn_enc" ||
            f == "eq_ignore_case" || f == "matches" || f == "match_indices" || f == "rmatch_indices" || f == "trim_start_matches" ||
            f == "trim_end_matches" || f == "lines" || f == "split_whitespace")
            return record_padded_extra(pg, psk, ssk, op, f, a, na, clear, err);
        tbh::FheString s = ssk.input_string(a[0]);
        if (f == "len") { output_radix(pg, psk.len(s)); return true; }
        if (f == "is_empty") { pg.output(psk.is_empty(s)); return true; }
        if (f == "trim_start") { output_string(pg, psk.trim_start(s)); return true; }
        if (f == "trim_end") { output_string(pg, psk.trim_end(s)); return true; }
        if (f == "trim") { output_string(pg, psk.trim(s)); return true; }
        if (f == "strip_prefix" || f == "strip_suffix") {
            if (!clear) { err = op + ": needs a clear pattern"; return false; }
            auto r = f == "strip_prefix" ? psk.strip_prefix(s, cl) : psk.strip_suffix(s, cl);
            pg.output(r.first);
            output_string(pg, r.second);
            return true;
        }
        if (f == "repeat") { if (!need(2)) return false; output_string(pg, psk.repeat(s, a[1])); return true; }
        if (!need(2)) return false;
        tbh::FheString t = ssk.input_string(a[1]);
        if (f == "eq") pg.output(psk.eq(s, t));
        else if (f == "ne") pg.output(psk.ne(s, t));
        else if (f == "lt") pg.output(psk.lt(s, t));
        else if (f == "le") pg.output(psk.le(s, t));
        else if (f == "gt") pg.output(psk.gt(s, t));
        else if (f == "ge") pg.output(psk.ge(s, t));
        else if (f == "contains") pg.output(psk.contains(s, t));
        else if (f == "starts_with") pg.output(psk.starts_with(s, t));
        else if (f == "ends_with") pg.output(psk.ends_with(s, t));
        else if (f == "concat") output_string(pg, psk.concat(s, t));
        else if (f == "find" || f == "rfind") { auto r = psk.find(s, t, f == "rfind"); pg.output(r.first); output_radix(pg, r.second); }
        else { err = "unknown padded string op: " + op; return false; }
        return true;
    }
    // ---- strings: a = {len_a[, len_b]}; with a non-empty `clear` the second operand is a clear (trivial) string ----------------------------------
    if (op.rfind("string_", 0) == 0) {
        if (!need(1)) return false;
        const std::string f = op.substr(7);
        tbh::FheString s = ssk.input_string(a[0]);
        if (f == "to_lowercase") { output_string(pg, ssk.to_lowercase(s)); return true; }
        if (f == "to_uppercase") { output_string(pg, ssk.to_uppercase(s)); return true; }
        tbh::FheString t;
        if (clear) t = ssk.trivial_string(cl);
        else { if (!need(2)) return false; t = ssk.input_string(a[1]); }
        if (f == "eq") pg.output(ssk.eq(s, t));
        else if (f == "ne") pg.output(ssk.ne(s, t));
        else if (f == "lt") pg.output(ssk.lt(s, t));
        else if (f == "le") pg.output(ssk.le(s, t));
        else if (f == "gt") pg.output(ssk.gt(s, t));
        else if (f == "ge") pg.output(ssk.ge(s, t));
        else if (f == "eq_ignore_case") pg.output(ssk.eq_ignore_case(s, t));
        else if (f == "contains") pg.output(ssk.contains(s, t));
        else if (f == "starts_with") pg.output(ssk.starts_with(s, t));
        else if (f == "ends_with") pg.output(ssk.ends_with(s, t));
        else if (f == "find") { auto r = ssk.find(s, t); pg.output(r.first); output_radix(pg, r.second); }
        else if (f == "rfind") { auto r = ssk.rfind(s, t); pg.output(r.first); output_radix(pg, r.second); }
        else if (f == "find_windows") {           // multi-GPU shard: first match among windows [a[2], a[3]) as a global index
            if (!need(4)) return false;
            if (a[2] > a[3]) { err = "find_windows: bad window range"; return false; }
            auto r = ssk.find_range(s, t, a[2], a[3]); pg.output(r.first); output_radix(pg, r.second);
        }
        else if (f == "cmp_sign") pg.output(ssk.compare_sign(s, t));     // multi-GPU shard of lt / le / gt / ge: the range's sign block
        else if (f == "contains_windows") {
            // multi-GPU shard: match flag OR-reduced over windows [a[2], a[3]) only -> one boolean block
            if (!need(4)) return false;
            const size_t nwin = t.len() <= s.len() ? s.len() - t.len() + 1 : 0;
            if (a[3] > nwin || a[2] >= a[3]) { err = "contains_windows: bad window range"; return false; }
            std::vector<tbh::Ct> mine = ssk.window_matches(s, t, a[2], a[3]);
            pg.output(isk.is_at_least_one_comparisons_block_true(mine));
        }
        else { err = "unknown string op: " + op; return false; }
        return true;
    }
    err = "unknown op: " + op;
    return false;
}

// frees the device copy of a program on the device it was uploaded to (no context needed: the owner may already be gone)
void release_device_state(tfhe_b200_program &h) {
    if (h.device < 0) return;
    DeviceGuard g(h.device);
    for (DevBuf *b : {&h.d_luts, &h.d_lin, &h.d_terms, &h.d_pbs_in, &h.d_pbs_out, &h.d_pbs_lut, &h.d_arena, &h.d_out_slots, &h.d_out_rows}) b->release();
    if (h.ev0) cudaEventDestroy(h.ev0);
    if (h.ev1) cudaEventDestroy(h.ev1);
    if (h.arena_done) cudaEventDestroy(h.arena_done);
    h.ev0 = h.ev1 = h.arena_done = nullptr;
    h.owner_id = 0;
    h.device = -1;
}

bool same_params(const tfhe_b200_params &q, const tbh::Params &p) {
    return q.lwe_dim == p.lwe_dim && q.glwe_dim == p.glwe_dim && q.poly_size == p.poly_size && q.pbs_base_log == p.pbs_base_log &&
           q.pbs_level == p.pbs_level && q.ks_base_log == p.ks_base_log && q.ks_level == p.ks_level &&
           q.grouping_factor == p.grouping_factor && q.msg_mod == p.msg_mod && q.carry_mod == p.carry_mod;
}

// first run on this context: upload the program (accumulators, instruction arrays) and size its arena.  A program bound to another
// context is re-bound (its old device copy is dropped); `owner_id` is only set once every upload has succeeded.
int bind_program(tfhe_b200_ctx *c, tfhe_b200_program *h) {
    if (h->owner_id == c->id) return 0;
    release_device_state(*h);
    const tbh::Program &pg = *h->prog;
    cudaStream_t s = c->stream;
    const size_t L = c->big_len();
    h->device = c->device;            // from here on release_device_state() knows where the partial uploads live
    TB_CUDA(cudaEventCreate(&h->ev0));
    TB_CUDA(cudaEventCreate(&h->ev1));
    TB_CUDA(cudaEventCreateWithFlags(&h->arena_done, cudaEventDisableTiming));
    std::vector<uint64_t> accs(std::max<size_t>(h->luts->size(), 1) * h->p.lut_len());
    for (size_t u = 0; u < h->luts->size(); ++u) h->luts->fill_accumulator(uint32_t(u), accs.data() + u * h->p.lut_len());
    TB_CUDA(h->d_luts.reserve(accs.size() * 8));
    TB_CUDA(cudaMemcpyAsync(h->d_luts.p, accs.data(), accs.size() * 8, cudaMemcpyHostToDevice, s));
    std::vector<tbk::LinInstr> lin;
    std::vector<uint32_t> pin, pout, plut;
    for (auto &l : pg.levels()) {
        for (auto &i : l.lin) lin.push_back({i.out_slot, i.term_begin, i.term_end, 0u, i.body_add});
        for (auto &j : l.pbs) { pin.push_back(j.in_slot); pout.push_back(j.out_slot); plut.push_back(j.lut); }
    }
    std::vector<tbk::LinTerm> terms;
    for (auto &t : pg.terms()) terms.push_back({t.slot, 0u, t.coef});
    auto up = [&](DevBuf &b, const void *src, size_t bytes) -> cudaError_t {
        cudaError_t e = b.reserve(std::max<size_t>(bytes, 16));
        if (e != cudaSuccess || bytes == 0) return e;
        return cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, s);
    };
    TB_CUDA(up(h->d_lin, lin.data(), lin.size() * sizeof(tbk::LinInstr)));
    TB_CUDA(up(h->d_terms, terms.data(), terms.size() * sizeof(tbk::LinTerm)));
    TB_CUDA(up(h->d_pbs_in, pin.data(), pin.size() * 4));
    TB_CUDA(up(h->d_pbs_out, pout.data(), pout.size() * 4));
    TB_CUDA(up(h->d_pbs_lut, plut.data(), plut.size() * 4));
    TB_CUDA(up(h->d_out_slots, pg.outputs().data(), pg.outputs().size() * 4));
    TB_CUDA(h->d_out_rows.reserve(std::max<size_t>(pg.outputs().size(), 1) * L * 8));
    TB_CUDA(h->d_arena.reserve(std::max<size_t>(pg.n_slots(), 1) * L * 8));
    TB_CUDA(cudaStreamSynchronize(s));   // the staging vectors above go out of scope
    h->owner_id = c->id;
    return 0;
}

// The shard plan of a level: a level of w PBS jobs is split across `world` ranks when w > min_shard_width (and world > 1); rank `rank`
// then runs jobs [lo, hi) of it (tbc::shard_range, possibly empty).  Every other level is replicated: every rank runs [0, w).  It depends
// only on (program, world, min_shard_width), so all ranks agree on it without talking.
bool level_share(const tfhe_b200_program *h, size_t lv, uint32_t rank, uint32_t world, uint64_t min_shard_width, size_t &lo, size_t &hi) {
    const size_t w = h->pbs_off[lv + 1] - h->pbs_off[lv];
    const bool split = world > 1 && w > min_shard_width;
    lo = 0; hi = w;
    if (split) tbc::shard_range(w, rank, world, lo, hi);
    return split;
}

// {split levels, largest share in rows (the exchange's max_rows), rows each rank receives over all split levels}
void shard_plan(const tfhe_b200_program *h, uint32_t world, uint64_t min_shard_width, uint64_t out[3]) {
    out[0] = out[1] = out[2] = 0;
    for (size_t lv = 0; lv + 1 < h->pbs_off.size(); ++lv) {
        size_t lo, hi;
        if (!level_share(h, lv, 0, world, min_shard_width, lo, hi)) continue;   // rank 0 has the largest share
        out[0] += 1;
        out[1] = std::max<uint64_t>(out[1], hi - lo);
        out[2] += h->pbs_off[lv + 1] - h->pbs_off[lv];
    }
}

// one rank of a run: its context, its program (bound to that context), its exchange (nullptr: an unsharded run) and its output rows
struct Member { tfhe_b200_ctx *c; tfhe_b200_program *h; tfhe_b200_exchange *ex; uint64_t *d_out; };

// Enqueues every level of the program on stream `s` for each of the `n` members: inputs are already in arena rows [0, n_inputs); the output
// rows end up in each member's d_out.  n == 1 without exchange: the plain run.  n == 1 with an exchange: rank ex->rank of a world of one
// process per GPU.  n == world > 1: every rank of one GPU, each level's shares enqueued rank after rank, then one cooperative scatter.
// A split level runs the linear instructions in full, the keyswitch and PBS of the member's share only (the PBS writes its rows
// contiguously into the exchange's send area), then the scatter that puts every share's rows into every member's arena.
int enqueue_levels(const Member *m, uint32_t n, uint64_t min_shard_width, cudaStream_t s) {
    const tbh::Program &pg = *m[0].h->prog;
    const uint32_t world = m[0].ex ? m[0].ex->world : 1;
    size_t max_w = 0;
    for (auto &l : pg.levels()) max_w = std::max(max_w, l.pbs.size());
    std::deque<tbc::StreamOrder> scratch;     // every member context's d_small and keyswitch digits, released when the levels are enqueued
    for (uint32_t i = 0; i < n; ++i) {
        scratch.emplace_back(m[i].c->scratch_done, s);
        TB_CUDA(scratch.back().wait);
        TB_CUDA(cudaEventRecord(m[i].h->ev0, s));
        TB_CUDA(m[i].c->d_small.reserve_on(std::max<size_t>(max_w, 1) * m[i].c->small_len() * 8, s));
    }
    std::vector<tfhe_b200_exchange *> exs(n);
    std::vector<const uint32_t *> out_slots(n);
    std::vector<uint64_t *> arenas(n);
    for (size_t lv = 0; lv < pg.levels().size(); ++lv) {
        const uint32_t l0 = m[0].h->lin_off[lv], l1 = m[0].h->lin_off[lv + 1], p0 = m[0].h->pbs_off[lv], p1 = m[0].h->pbs_off[lv + 1];
        bool split = false;
        for (uint32_t i = 0; i < n; ++i) {
            tfhe_b200_ctx *c = m[i].c;
            tfhe_b200_program *h = m[i].h;
            const size_t L = c->big_len();
            uint64_t *arena = (uint64_t *)h->d_arena.p;
            if (l1 > l0) {
                TB_CUDA(tbk::launch_linear(arena, (const tbk::LinInstr *)h->d_lin.p + l0, (const tbk::LinTerm *)h->d_terms.p, int(l1 - l0), int(L), s));
                c->launches += 1;
            }
            size_t lo, hi;
            split = level_share(h, lv, m[i].ex ? m[i].ex->rank : 0, world, min_shard_width, lo, hi);
            if (hi > lo) {
                const size_t w = hi - lo;
                const bool fused = tbc::fused_supported(c);
                if (tbc::do_keyswitch(c, arena, (uint64_t *)c->d_small.p, w, s, (const uint32_t *)h->d_pbs_in.p + p0 + lo, nullptr, fused)) return 1;
                if (tbc::do_pbs(c, (const uint64_t *)c->d_small.p, (const uint32_t *)h->d_pbs_lut.p + p0 + lo, (const uint64_t *)h->d_luts.p,
                                split ? tbc::exchange_next_send_area(m[i].ex) : arena, w, c->p.lwe_dim, s,
                                split ? nullptr : (const uint32_t *)h->d_pbs_out.p + p0, fused))
                    return 1;
            }
            exs[i] = m[i].ex;
            out_slots[i] = (const uint32_t *)h->d_pbs_out.p + p0;
            arenas[i] = arena;
        }
        if (split) {
            if (n > 1 ? tbc::exchange_scatter_group(exs.data(), n, p1 - p0, out_slots.data(), arenas.data(), s)
                      : tbc::exchange_scatter(exs[0], p1 - p0, out_slots[0], arenas[0], s))
                return 1;
        }
    }
    for (uint32_t i = 0; i < n; ++i) {
        TB_CUDA(cudaEventRecord(m[i].h->ev1, s));
        if (!pg.outputs().empty()) {   // gather the output rows on the device
            TB_CUDA(tbk::launch_gather_rows((uint64_t *)m[i].h->d_arena.p, (const uint32_t *)m[i].h->d_out_slots.p, m[i].d_out,
                                            (int)pg.outputs().size(), (int)m[i].c->big_len(), s));
            m[i].c->launches += 1;
        }
    }
    return 0;
}

// everything a sharded run checks about one rank before it enqueues anything
int check_sharded_member(const char *who, tfhe_b200_ctx *c, tfhe_b200_program *h, tfhe_b200_exchange *ex, const uint64_t *d_inputs,
                         uint64_t *d_outputs, uint64_t min_shard_width) {
    const std::string w = who;
    if (!c || !h || !ex) return fail(w + ": null argument");
    const tbh::Program &pg = *h->prog;
    if ((pg.n_inputs() && !d_inputs) || (!pg.outputs().empty() && !d_outputs)) return fail(w + ": null buffer");
    if (!same_params(c->p, h->p)) return fail(w + ": program was recorded for other parameters than the context");
    if (ex->ctx != c) return fail(w + ": the exchange of rank " + std::to_string(ex->rank) + " belongs to another context");
    if (!ex->attached) return fail(w + ": exchange peers not attached yet (tfhe_b200_exchange_attach)");
    uint64_t plan[3];
    shard_plan(h, ex->world, min_shard_width, plan);
    if (plan[1] > ex->max_rows)
        return fail(w + ": " + h->op + " at world " + std::to_string(ex->world) + " and min_shard_width " + std::to_string(min_shard_width) +
                    " needs an exchange of max_rows >= " + std::to_string(plan[1]) + ", this one holds " + std::to_string(ex->max_rows));
    return 0;
}

}  // namespace

extern "C" {

int tfhe_b200_program_build(const tfhe_b200_params *params, const char *op, const uint64_t *args, size_t n_args,
                            const char *clear_operand, tfhe_b200_program **out) {
    if (!out) return fail("null out pointer");
    *out = nullptr;
    if (!params || !op) return fail("null argument");
    if (params->msg_mod < 2 || params->carry_mod < 1 || (params->poly_size % (params->msg_mod * params->carry_mod)) != 0)
        return fail("bad message / carry modulus");
    auto h = std::make_unique<tfhe_b200_program>();
    h->p = to_host_params(*params);
    h->luts = std::make_unique<tbh::LutRegistry>(h->p);
    h->prog = std::make_unique<tbh::Program>(h->p, *h->luts);
    h->op = op;
    std::string err;
    try {
        if (!record(*h, op, args, n_args, clear_operand, err)) return fail(err);
    } catch (const std::exception &e) {
        return fail(std::string(op) + ": " + e.what());
    }
    uint32_t lo = 0, po = 0;
    for (auto &l : h->prog->levels()) {
        h->lin_off.push_back(lo); h->pbs_off.push_back(po);
        lo += uint32_t(l.lin.size()); po += uint32_t(l.pbs.size());
    }
    h->lin_off.push_back(lo); h->pbs_off.push_back(po);
    *out = h.release();
    return 0;
}

int tfhe_b200_program_destroy(tfhe_b200_program *h) {
    if (!h) return 0;
    release_device_state(*h);
    delete h;
    return 0;
}

/* counts[8] = {n_inputs, n_outputs, n_slots, n_levels, n_lin, n_terms, n_pbs, n_luts}; counts[8] = trivial PBS folded on the host */
int tfhe_b200_program_counts(const tfhe_b200_program *h, uint64_t counts[9]) {
    if (!h || !counts) return fail("null argument");
    const tbh::Program &pg = *h->prog;
    counts[0] = pg.n_inputs(); counts[1] = pg.outputs().size(); counts[2] = pg.n_slots(); counts[3] = pg.levels().size();
    counts[4] = h->lin_off.back(); counts[5] = pg.terms().size(); counts[6] = h->pbs_off.back(); counts[7] = h->luts->size();
    counts[8] = pg.n_trivial_pbs();
    return 0;
}

/* Copies the recorded program out (for inspection and for executing it with another backend, e.g. the CPU oracle in tests).
 * Array sizes follow tfhe_b200_program_counts.  Any pointer may be NULL to skip that part. */
int tfhe_b200_program_copy(const tfhe_b200_program *h, uint32_t *level_lin_off, uint32_t *level_pbs_off, uint32_t *lin_out_tb_te,
                           uint64_t *lin_body, uint32_t *term_slot, int64_t *term_coef, uint32_t *pbs_in_out_lut,
                           uint64_t *lut_tables, uint64_t *lut_degrees, uint32_t *outputs, uint64_t *output_degree_noise) {
    if (!h) return fail("null argument");
    const tbh::Program &pg = *h->prog;
    if (level_lin_off) std::copy(h->lin_off.begin(), h->lin_off.end(), level_lin_off);
    if (level_pbs_off) std::copy(h->pbs_off.begin(), h->pbs_off.end(), level_pbs_off);
    size_t li = 0, pi = 0;
    for (auto &l : pg.levels()) {
        for (auto &i : l.lin) {
            if (lin_out_tb_te) { lin_out_tb_te[3 * li] = i.out_slot; lin_out_tb_te[3 * li + 1] = i.term_begin; lin_out_tb_te[3 * li + 2] = i.term_end; }
            if (lin_body) lin_body[li] = i.body_add;
            ++li;
        }
        for (auto &j : l.pbs) {
            if (pbs_in_out_lut) { pbs_in_out_lut[3 * pi] = j.in_slot; pbs_in_out_lut[3 * pi + 1] = j.out_slot; pbs_in_out_lut[3 * pi + 2] = j.lut; }
            ++pi;
        }
    }
    for (size_t t = 0; t < pg.terms().size(); ++t) {
        if (term_slot) term_slot[t] = pg.terms()[t].slot;
        if (term_coef) term_coef[t] = pg.terms()[t].coef;
    }
    for (size_t u = 0; u < h->luts->size(); ++u) {
        if (lut_tables) std::copy(h->luts->lut(u).table.begin(), h->luts->lut(u).table.end(), lut_tables + u * h->p.total_mod());
        if (lut_degrees) lut_degrees[u] = h->luts->lut(u).degree;
    }
    for (size_t o = 0; o < pg.outputs().size(); ++o) {
        if (outputs) outputs[o] = pg.outputs()[o];
        if (output_degree_noise) { output_degree_noise[2 * o] = pg.output_meta()[o].degree; output_degree_noise[2 * o + 1] = pg.output_meta()[o].noise; }
    }
    return 0;
}

/* Accumulators of the program's LUTs as ServerKey::generate_lookup_table would build them (n_luts x (k+1)*N words). */
int tfhe_b200_program_accumulators(const tfhe_b200_program *h, uint64_t *accs) {
    if (!h || !accs) return fail("null argument");
    for (size_t u = 0; u < h->luts->size(); ++u) h->luts->fill_accumulator(uint32_t(u), accs + u * h->p.lut_len());
    return 0;
}

/* Executes the program on `ctx` (its keys must be uploaded).  inputs: n_inputs x (k*N+1) words (host), in the order the
 * operation declares its operands; outputs: n_outputs x (k*N+1) words (host). */
int tfhe_b200_program_run(tfhe_b200_ctx *c, tfhe_b200_program *h, const uint64_t *inputs, uint64_t *outputs) {
    if (!c || !h) return fail("null argument");
    const tbh::Program &pg = *h->prog;
    if ((pg.n_inputs() && !inputs) || (!pg.outputs().empty() && !outputs)) return fail("null buffer");
    if (!same_params(c->p, h->p)) return fail("program was recorded for other parameters than the context");
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    cudaStream_t s = c->stream;
    const size_t L = c->big_len();
    if (bind_program(c, h)) return 1;
    tbc::StreamOrder arena(h->arena_done, s);     // a run_device of this program may be pending on another stream
    TB_CUDA(arena.wait);
    if (pg.n_inputs()) TB_CUDA(cudaMemcpyAsync(h->d_arena.p, inputs, (size_t)pg.n_inputs() * L * 8, cudaMemcpyHostToDevice, s));
    const Member m{c, h, nullptr, (uint64_t *)h->d_out_rows.p};
    if (enqueue_levels(&m, 1, 0, s)) return 1;
    if (!pg.outputs().empty())     // one copy back
        TB_CUDA(cudaMemcpyAsync(outputs, h->d_out_rows.p, pg.outputs().size() * L * 8, cudaMemcpyDeviceToHost, s));
    TB_CUDA(cudaStreamSynchronize(s));
    TB_CUDA(cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
    return 0;
}

/* The same on DEVICE buffers of the context's GPU, enqueued on `cuda_stream` (NULL = the context's own stream) WITHOUT synchronising:
 * d_inputs n_inputs x (k*N+1) words, d_outputs n_outputs x (k*N+1) words.  This is what chains a rank's share of a sharded string
 * operation, the exchange of the narrow-end blocks and the finishing program without a host round trip (multi_gpu.py).
 * Calls on other streams may overlap it: the context's keyswitch scratch and the program's arena are taken in enqueue order (StreamOrder). */
int tfhe_b200_program_run_device(tfhe_b200_ctx *c, tfhe_b200_program *h, const uint64_t *d_inputs, uint64_t *d_outputs, void *cuda_stream) {
    if (!c || !h) return fail("null argument");
    const tbh::Program &pg = *h->prog;
    if ((pg.n_inputs() && !d_inputs) || (!pg.outputs().empty() && !d_outputs)) return fail("null buffer");
    if (!same_params(c->p, h->p)) return fail("program was recorded for other parameters than the context");
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    const size_t L = c->big_len();
    if (bind_program(c, h)) return 1;
    tbc::StreamOrder arena(h->arena_done, s);
    TB_CUDA(arena.wait);
    if (pg.n_inputs()) TB_CUDA(cudaMemcpyAsync(h->d_arena.p, d_inputs, (size_t)pg.n_inputs() * L * 8, cudaMemcpyDeviceToDevice, s));
    h->last_ms = -1.f;    // not synchronised: tfhe_b200_program_last_ms reads the events on demand
    const Member m{c, h, nullptr, d_outputs};
    return enqueue_levels(&m, 1, 0, s);
}

/* {split levels, largest share in rows, rows each rank receives} of a sharded run at (world, min_shard_width); pure host arithmetic. */
int tfhe_b200_program_shard_plan(const tfhe_b200_program *h, uint32_t world, uint64_t min_shard_width, uint64_t out[3]) {
    if (!h || !out) return fail("null argument");
    if (world < 1) return fail("program_shard_plan: world must be >= 1");
    shard_plan(h, world, min_shard_width, out);
    return 0;
}

/* Rank `rank`'s PBS jobs of level `level` in a sharded run: out = {lo, hi, split}, jobs [lo, hi) counted from the level's first job.
 * A replicated level (split = 0) gives [0, width) to every rank. */
int tfhe_b200_program_level_share(const tfhe_b200_program *h, uint32_t level, uint32_t rank, uint32_t world, uint64_t min_shard_width,
                                  uint64_t out[3]) {
    if (!h || !out) return fail("null argument");
    if (world < 1 || rank >= world) return fail("program_level_share: need world >= 1 and rank < world");
    if ((size_t)level + 1 >= h->pbs_off.size()) return fail("program_level_share: no level " + std::to_string(level));
    size_t lo, hi;
    out[2] = level_share(h, level, rank, world, min_shard_width, lo, hi);
    out[0] = lo; out[1] = hi;
    return 0;
}

/* One rank of a program run across the ranks of `ex` (one process per GPU): levels wider than min_shard_width are split, every rank runs
 * its share and the scatter exchange hands every row to every rank; the other levels run in full on every rank.  Every rank passes all
 * inputs and receives all outputs; device buffers, enqueued on `cuda_stream` (NULL = the context's stream) without synchronising. */
int tfhe_b200_program_run_sharded(tfhe_b200_ctx *c, tfhe_b200_program *h, tfhe_b200_exchange *ex, const uint64_t *d_inputs, uint64_t *d_outputs,
                                  uint64_t min_shard_width, void *cuda_stream) {
    if (check_sharded_member("program_run_sharded", c, h, ex, d_inputs, d_outputs, min_shard_width)) return 1;
    if (ex->shares_device)
        return fail("program_run_sharded: ranks that share a GPU must use tfhe_b200_program_run_sharded_group (kernels that wait on one another "
                    "cannot be separate launches on one device)");
    const tbh::Program &pg = *h->prog;
    std::lock_guard<std::mutex> lk(c->mu);
    DeviceGuard g(c->device);
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    if (bind_program(c, h)) return 1;
    tbc::StreamOrder arena(h->arena_done, s);
    TB_CUDA(arena.wait);
    if (pg.n_inputs()) TB_CUDA(cudaMemcpyAsync(h->d_arena.p, d_inputs, (size_t)pg.n_inputs() * c->big_len() * 8, cudaMemcpyDeviceToDevice, s));
    h->last_ms = -1.f;
    const Member m{c, h, ex, d_outputs};
    return enqueue_levels(&m, 1, min_shard_width, s);
}

/* Every rank of one GPU in one call on one stream (ctxs[r], progs[r], exs[r]: rank r's context, its own program object -- a program binds
 * to one context -- and its exchange, attached with tfhe_b200_exchange_attach_local).  Per split level every rank's share is enqueued,
 * then one cooperative scatter serves all ranks. */
int tfhe_b200_program_run_sharded_group(tfhe_b200_ctx *const *ctxs, tfhe_b200_program *const *progs, tfhe_b200_exchange *const *exs, uint32_t world,
                                        const uint64_t *const *d_inputs, uint64_t *const *d_outputs, uint64_t min_shard_width, void *cuda_stream) {
    const char *who = "program_run_sharded_group";
    if (!ctxs || !progs || !exs || !d_inputs || !d_outputs || world < 1) return fail(std::string(who) + ": null argument");
    for (uint32_t r = 0; r < world; ++r) {
        if (check_sharded_member(who, ctxs[r], progs[r], exs[r], d_inputs[r], d_outputs[r], min_shard_width)) return 1;
        if (exs[r]->world != world || exs[r]->rank != r)
            return fail(std::string(who) + ": exchange " + std::to_string(r) + " is rank " + std::to_string(exs[r]->rank) + " of " +
                        std::to_string(exs[r]->world) + ", not rank " + std::to_string(r) + " of " + std::to_string(world));
        if (exs[0]->peer[r] != exs[r]->local.p)
            return fail(std::string(who) + ": exchange " + std::to_string(r) + " is not attached to exchange 0 (tfhe_b200_exchange_attach_local)");
        if (ctxs[r]->device != ctxs[0]->device)
            return fail(std::string(who) + ": rank " + std::to_string(r) + " is on device " + std::to_string(ctxs[r]->device) + ", rank 0 on device " +
                        std::to_string(ctxs[0]->device) + ": a group runs on one GPU (use tfhe_b200_program_run_sharded, one process per GPU)");
        if (progs[r]->op != progs[0]->op || progs[r]->pbs_off != progs[0]->pbs_off || progs[r]->lin_off != progs[0]->lin_off ||
            !same_params(ctxs[r]->p, progs[0]->p))
            return fail(std::string(who) + ": rank " + std::to_string(r) + " runs another program or parameter set than rank 0");
        for (uint32_t q = 0; q < r; ++q)
            if (progs[q] == progs[r] || ctxs[q] == ctxs[r])
                return fail(std::string(who) + ": ranks " + std::to_string(q) + " and " + std::to_string(r) +
                            " share a context or a program object (each rank needs its own; a program binds to one context)");
    }
    const tbh::Program &pg = *progs[0]->prog;
    std::vector<std::unique_lock<std::mutex>> locks;
    for (uint32_t r = 0; r < world; ++r) locks.emplace_back(ctxs[r]->mu);
    DeviceGuard g(ctxs[0]->device);
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : ctxs[0]->stream;
    std::vector<Member> m(world);
    for (uint32_t r = 0; r < world; ++r) {
        if (bind_program(ctxs[r], progs[r])) return 1;
        m[r] = Member{ctxs[r], progs[r], exs[r], d_outputs[r]};
    }
    std::deque<tbc::StreamOrder> arena;
    for (uint32_t r = 0; r < world; ++r) {
        arena.emplace_back(progs[r]->arena_done, s);
        TB_CUDA(arena.back().wait);
        if (pg.n_inputs())
            TB_CUDA(cudaMemcpyAsync(progs[r]->d_arena.p, d_inputs[r], (size_t)pg.n_inputs() * ctxs[r]->big_len() * 8, cudaMemcpyDeviceToDevice, s));
        progs[r]->last_ms = -1.f;
    }
    return enqueue_levels(m.data(), world, min_shard_width, s);
}

/* Device time (ms, CUDA events on the context stream) of the kernels of the last tfhe_b200_program_run. */
int tfhe_b200_program_last_ms(const tfhe_b200_program *h, float *ms) {
    if (!h || !ms) return fail("null argument");
    if (h->last_ms < 0.f && h->ev1) {   // last run was tfhe_b200_program_run_device: wait for its end event
        DeviceGuard g(h->device);
        TB_CUDA(cudaEventSynchronize(h->ev1));
        TB_CUDA(cudaEventElapsedTime(ms, h->ev0, h->ev1));
        return 0;
    }
    *ms = h->last_ms;
    return 0;
}

}  // extern "C"
