"""The host layer at every message / carry modulus the engine accepts (CPU, no GPU).

Every op of the program API (include/tfhe_b200.h, tfhe_b200_program_build) is recorded with the moduli of each of the 36 classic
PARAM_MESSAGE_<m>_CARRY_<c>_KS_PBS sets and executed noise-free on plaintexts against Python semantics.  The rule: an op returns the
right value on every input, or it refuses with NativeError when it is built.  It never returns a wrong value.  Which ops each set
refuses is pinned in REFUSED, so a change in coverage shows up as a failure.

Inputs include all-max blocks, x = m^B - 1 plus 0 and plus 1, every block degree from m - 1 to total_mod - 1 for the propagating ops,
chars 0x00, 0x7f and 0xff, and the string pairs whose packed block equalities used to overflow.  The last tests run a few of these
programs with the CPU oracle's real KS-PBS on the toy keys, with the moduli overridden."""
from __future__ import annotations

import numpy as np
import pytest

from fhe_string_bounty_b200 import NativeError, _native as N
from fhe_string_bounty_b200.host import Program
from helpers import engine_params
from test_padded_split_replace import digits_for, max_matches, rs_replacen, rs_split_once, rs_splitn

SETS = list(N._CLASSIC_SETS)
NB = 3                                        # radix blocks of the integer ops
WS = b" \t\n\r\x0b\x0c"                       # char::is_whitespace restricted to ASCII


# ---- noise-free execution of a batch of inputs -------------------------------------------------------------------------------------
def simulate_batch(ir, rows, total_mod):
    """helpers.simulate_program_clear over many input rows at once: rows [batch, n_inputs] -> outputs [batch, n_outputs].  A slot holds
    its value modulo 2 * total_mod; a PBS operand at or above total_mod reaches the padding bit and returns -f(x - total_mod)."""
    T, M = total_mod, 2 * total_mod
    delta = (1 << 63) // T
    rows = np.asarray(rows, dtype=np.int64).reshape(-1, ir.n_inputs)
    val = np.zeros((ir.n_slots, rows.shape[0]), dtype=np.int64)
    val[: ir.n_inputs] = rows.T
    tables = ir.lut_tables.astype(np.int64)
    for lv in range(len(ir.level_lin_off) - 1):
        for li in range(int(ir.level_lin_off[lv]), int(ir.level_lin_off[lv + 1])):
            out, tb, te = (int(v) for v in ir.lin[li])
            body = int(ir.lin_body[li])
            assert body % delta == 0, "plaintext bodies are multiples of delta"
            acc = np.full(rows.shape[0], body // delta, dtype=np.int64)
            for t in range(tb, te):
                acc += int(ir.term_coef[t]) * val[int(ir.term_slot[t])]
            val[out] = acc % M
        p0, p1 = int(ir.level_pbs_off[lv]), int(ir.level_pbs_off[lv + 1])
        if p1 > p0:
            src, dst, lut = ir.pbs[p0:p1, 0], ir.pbs[p0:p1, 1], ir.pbs[p0:p1, 2]
            x = val[src]
            t = tables[lut[:, None], x % T]
            val[dst] = np.where(x >= T, (-t) % M, t)
    return val[ir.outputs].T


# ---- plaintext encodings ---------------------------------------------------------------------------------------------------------
def radix_digits(v, m, n):
    return [(v // m**i) % m for i in range(n)]


def bits_of(m):
    return m.bit_length() - 1


def str_blocks(s: bytes, m):
    """a char is ceil(8 / log2 m) little-endian blocks of log2 m bits (host/strings.h blocks_per_char)"""
    b = bits_of(m)
    return [(ch >> (b * k)) & (m - 1) for ch in s for k in range(-(-8 // b))]


def pad(s: bytes, cap):
    return s + b"\0" * (cap - len(s))


class Case:
    """one recorded program and its rows: (inputs, expected outputs); `key` names it in REFUSED"""

    def __init__(self, key, op, args, clear=None, rows=None, expect=None):
        self.key, self.op, self.args, self.clear = key, op, tuple(int(a) for a in args), clear
        self.rows = rows or []           # list of (inputs, expected outputs)
        self.expect = expect             # alternative: f(program) -> rows, when the expected length depends on the program's outputs


def _cmp(x, y):
    return {"eq": x == y, "ne": x != y, "lt": x < y, "le": x <= y, "gt": x > y, "ge": x >= y}


# ---- the op list --------------------------------------------------------------------------------------------------------------
def integer_cases(m, c, rng):
    T, R = m * c, m**NB
    vals = sorted({0, 1, m - 1, m, R // 2, R - 2, R - 1, *(int(v) for v in rng.integers(0, R, size=3))})
    pairs = [(x, y) for x in vals for y in vals]
    enc = lambda x: radix_digits(x, m, NB)
    for f in ("eq", "ne", "lt", "le", "gt", "ge"):
        yield Case(f"radix_{f}", f"radix_{f}", (NB,), rows=[(enc(x) + enc(y), [int(_cmp(x, y)[f])]) for x, y in pairs])
    yield Case("radix_eq_packed", "radix_eq_packed", (NB,), rows=[(enc(x) + enc(y), [int(x == y)]) for x, y in pairs])
    yield Case("radix_add", "radix_add", (NB,), rows=[(enc(x) + enc(y), enc((x + y) % R)) for x, y in pairs])
    for s in (0, 1, m, R // 2, R - 1, R, R + 5):
        key = "" if s < R else "/above"      # a scalar above the radix folds to a trivial result on the host
        for f, w in (("eq", lambda x: x == s), ("lt", lambda x: x < s), ("gt", lambda x: x > s)):
            yield Case(f"radix_scalar_{f}{key}", f"radix_scalar_{f}", (NB, s), rows=[(enc(x), [int(w(x))]) for x in vals])
    yield Case("radix_if_then_else", "radix_if_then_else", (NB,),
               rows=[([cnd] + enc(x) + enc(y), enc(x if cnd else y)) for x, y in pairs[::3] for cnd in (0, 1)])
    # the propagating ops at every block degree: blocks hold up to `d` (message plus carries), the value is sum b_i m^i mod m^NB
    for d in range(m - 1, T):
        blocks = [[d] * NB, [d, 0, d], [0, d, d], [d, d - 1 if d else 0, 1], [m - 1] * NB, [0] * NB]
        blocks += [list(rng.integers(0, d + 1, size=NB)) for _ in range(6)]
        value = lambda b: sum(int(v) * m**i for i, v in enumerate(b)) % R
        yield Case(f"radix_full_propagate@{d}", "radix_full_propagate", (NB, d), rows=[(list(b), enc(value(b))) for b in blocks])
        for f in ("eq", "ne", "lt", "le", "gt", "ge"):
            rows = [(list(a) + list(b), [int(_cmp(value(a), value(b))[f])]) for a in blocks for b in blocks[::2]]
            yield Case(f"radix_default_{f}@{d}", f"radix_default_{f}", (NB, d), rows=rows)


def shortint_and_bool_cases(m, c, rng):
    T = m * c
    f = [(3 * x + 1) % T for x in range(T)]
    yield Case("shortint_apply_lut", "shortint_apply_lut", [T] + f, rows=[(list(range(T)), f)])
    g = [(x * y + x + 1) % T for x in range(m) for y in range(m)]
    xs, ys = [x for x in range(m) for _ in range(m)], [y for _ in range(m) for y in range(m)]
    yield Case("shortint_bivariate_lut", "shortint_bivariate_lut", [m * m] + g, rows=[(xs + ys, g)])
    for n in (3, T + 1):
        rows = [[1] * n, [0] * n] + [[int(i != j) for i in range(n)] for j in (0, n // 2, n - 1)] + [[int(i == n - 1) for i in range(n)]]
        yield Case("bool_all_true", "bool_all_true", (n,), rows=[(r, [int(all(r))]) for r in rows])
        yield Case("bool_any_true", "bool_any_true", (n,), rows=[(r, [int(any(r))]) for r in rows])
    n = T - 1
    for want_all in (0, 1):
        yield Case("bool_sum_finish", "bool_sum_finish", (n, want_all), rows=[([s], [int(s == n if want_all else s != 0)]) for s in range(n + 1)])
    combos = [[a, b, d] for a in range(3) for b in range(3) for d in range(3)]            # least significant range first
    for want_less in (0, 1):
        for or_equal in (0, 1):
            def want(sg):
                top = next((v for v in reversed(sg) if v != 1), 1)
                return int(or_equal) if top == 1 else int(top == (0 if want_less else 2))
            yield Case("signs_finish", "signs_finish", (3, want_less, or_equal), rows=[(sg, [want(sg)]) for sg in combos])
    count = max(1, min(3, T // 2))
    rows = []
    for _ in range(12):
        flags = list(rng.integers(0, 2, size=count))
        idx = [int(v) for v in rng.integers(0, m**2, size=count)]
        first = next((i for i in range(count) if flags[i]), None)
        ins = [v for r in range(count) for v in [int(flags[r])] + radix_digits(idx[r], m, 2)]
        rows.append((ins, [int(first is not None)] + radix_digits(idx[first] if first is not None else 0, m, 2)))
    yield Case("find_combine", "find_combine", (count, 2), rows=rows)


# lengths (3, 2) and (2, 2); all-max chars, 0x00 / 0x7f neighbours, the pairs whose packed equality overflowed (3_0, 3_1, 8_0)
PAIRS_32 = [(b"zz~", b"zz"), (b"~zz", b"zz"), (b"abz", b"bz"), (b"aaa", b"aa"), (b"\x7f\x00\x01", b"\x00\x01"), (b"\xff\xff\xff", b"\xff\xff"),
            (b"xyz", b"ab"), (b"AbC", b"bc")]
PAIRS_22 = [(b"\x7f\x00", b"\x7f\x01"), (b"\x7f\x01", b"\x7f\x00"), (b"ab", b"ab"), (b"Ab", b"aB"), (b"\x00\x00", b"\x00\x00"),
            (b"\xff\xff", b"\xff\xfe"), (b"\xfe\xff", b"\xff\xfe"), (b"zz", b"ZZ")]


def _string_want(f, a, b):
    if f in ("find", "rfind"):
        pos = a.find(b) if f == "find" else a.rfind(b)
        return int(pos >= 0), max(pos, 0)
    return {"eq": a == b, "ne": a != b, "lt": a < b, "le": a <= b, "gt": a > b, "ge": a >= b, "eq_ignore_case": a.lower() == b.lower(),
            "contains": b in a, "starts_with": a.startswith(b), "ends_with": a.endswith(b)}[f]


def _index_digits(la, lb):
    W, d = la - lb + 1, 1
    while 4**d < max(W, 1):
        d += 1
    return d


def string_cases(m, c):
    S = lambda s: str_blocks(s, m)
    ops = ["eq", "ne", "lt", "le", "gt", "ge", "eq_ignore_case", "contains", "starts_with", "ends_with", "find", "rfind"]
    for pairs in (PAIRS_32, PAIRS_22):
        la, lb = len(pairs[0][0]), len(pairs[0][1])
        for f in ops:
            def out(a, b, f=f):
                w = _string_want(f, a, b)
                return [w[0]] + radix_digits(w[1], 4, _index_digits(la, lb)) if f in ("find", "rfind") else [int(w)]
            for suffix in ("", "_packed"):
                yield Case(f"string_{f}{suffix}", f"string_{f}{suffix}", (la, lb), rows=[(S(a) + S(b), out(a, b)) for a, b in pairs])
            if f != "eq_ignore_case":
                for a, b in (ab for ab in pairs if 0 not in ab[1]):      # a C string cannot hold a NUL char
                    yield Case(f"string_{f}/clear", f"string_{f}", (la,), clear=b.decode("latin-1"), rows=[(S(a), out(a, b))])
        for f in ("eq", "ne", "lt", "le", "contains"):
            rows = [(S(a0) + S(b0) + S(a1) + S(b1), [int(_string_want(f, a0, b0)), int(_string_want(f, a1, b1))])
                    for (a0, b0), (a1, b1) in zip(pairs, pairs[1:] + pairs[:1])]
            for suffix in ("", "_packed"):
                yield Case(f"string_{f}_many{suffix}", f"string_{f}_many{suffix}", (la, lb, 2), rows=rows)
    # lower / upper case, multi-GPU shards: one window range, and the sign block of a whole comparison
    words = [a for a, _ in PAIRS_32] + [b"@AZ", b"[`a", b"z{\x00"]
    yield Case("string_to_lowercase", "string_to_lowercase", (3,), rows=[(S(w), S(w.lower())) for w in words])
    yield Case("string_to_uppercase", "string_to_uppercase", (3,), rows=[(S(w), S(w.upper())) for w in words])
    rows = [(S(a) + S(b), [int(a[1:].startswith(b))] + radix_digits(1 if a[1:].startswith(b) else 0, 4, 1)) for a, b in PAIRS_32]
    yield Case("string_find_windows", "string_find_windows", (3, 2, 1, 2), rows=rows)
    yield Case("string_contains_windows", "string_contains_windows", (3, 2, 1, 2), rows=[(S(a) + S(b), [int(a[1:] == b)]) for a, b in PAIRS_32])
    yield Case("string_cmp_sign", "string_cmp_sign", (2, 2), rows=[(S(a) + S(b), [0 if a < b else 1 if a == b else 2]) for a, b in PAIRS_22])


def padded_cases(m, c):
    """the null-padded model (host/padded.h); programs are small, the expected output length comes from the program"""
    S = lambda s, cap: str_blocks(pad(s, cap), m)
    unary = [b"", b"a", b" x ", b"\t\n\x0b\x0c", b"\xff\xff\xff\xff", b"ab  "]
    cap = 4
    digits = lambda v, P: radix_digits(v, 4, P.n_outputs)
    yield Case("pstring_len", "pstring_len", (cap,), expect=lambda P: [(S(s, cap), digits(len(s), P)) for s in unary])
    yield Case("pstring_is_empty", "pstring_is_empty", (cap,), rows=[(S(s, cap), [int(not s)]) for s in unary])
    for f, op in (("trim_start", lambda s: s.lstrip(WS)), ("trim_end", lambda s: s.rstrip(WS)), ("trim", lambda s: s.strip(WS))):
        yield Case(f"pstring_{f}", f"pstring_{f}", (cap,), rows=[(S(s, cap), S(op(s), cap)) for s in unary])
    for pat in (b"a", b" x"):
        yield Case("pstring_strip_prefix", "pstring_strip_prefix", (cap,), clear=pat.decode(),
                   rows=[(S(s, cap), [int(s.startswith(pat))] + S(s[len(pat):] if s.startswith(pat) else s, cap)) for s in unary])
        yield Case("pstring_strip_suffix", "pstring_strip_suffix", (cap,), clear=pat.decode(),
                   rows=[(S(s, cap), [int(s.endswith(pat))] + S(s[:-len(pat)] if s.endswith(pat) else s, cap)) for s in unary])
    yield Case("pstring_repeat", "pstring_repeat", (2, 3), rows=[(S(s, 2), S(s * 3, 6)) for s in (b"", b"a", b"\xff\xff")])
    pairs = [(b"abab", b"ab"), (b"ab", b""), (b"", b""), (b"\xff\xff\xff", b"\xff\xff"), (b"aab", b"ab"), (b"b", b"abc"), (b"zz~", b"zz")]
    ca, cb = 4, 3
    for f in ("eq", "ne", "lt", "le", "gt", "ge", "contains", "starts_with", "ends_with"):
        yield Case(f"pstring_{f}", f"pstring_{f}", (ca, cb), rows=[(S(a, ca) + S(b, cb), [int(_string_want(f, a, b))]) for a, b in pairs])
    yield Case("pstring_concat", "pstring_concat", (ca, cb), rows=[(S(a, ca) + S(b, cb), S(a + b, ca + cb)) for a, b in pairs])
    for f in ("find", "rfind"):
        def rows_of(P, f=f):
            out = []
            for a, b in pairs:
                pos = a.find(b) if f == "find" else a.rfind(b)
                out.append((S(a, ca) + S(b, cb), [int(pos >= 0)] + radix_digits(max(pos, 0), 4, P.n_outputs - 1)))
            return out
        yield Case(f"pstring_{f}", f"pstring_{f}", (ca, cb), expect=rows_of)
    hays, pats, to, cp = [b"", b"aaa", b"aba", b"a,b"], [b"", b"a", b"ab"], b"<>", 2
    C = 3 + max_matches(3, 0) * 2
    yield Case("pstring_replace", "pstring_replace", (3, cp, 2),
               rows=[(S(s, 3) + S(p, cp) + S(to, 2), S(rs_replacen(s, p, to), C)) for s in hays for p in pats])
    C1 = 3 + 1 * 2
    yield Case("pstring_replacen", "pstring_replacen", (3, cp, 2, 1),
               rows=[(S(s, 3) + S(p, cp) + S(to, 2), S(rs_replacen(s, p, to, 1), C1)) for s in hays for p in pats])
    for name, n in (("pstring_split", None), ("pstring_splitn", 2)):
        Pn = max_matches(3, 0) + 1 if n is None else min(max_matches(3, 0) + 1, n)
        nd = digits_for(Pn)
        rows = []
        for s in hays:
            for p in pats:
                want = rs_splitn(s, p, n)
                rows.append((S(s, 3) + S(p, cp), radix_digits(len(want), 4, nd) + sum((S(w, 3) for w in want + [b""] * (Pn - len(want))), [])))
        yield Case(name, name, (3, cp) if n is None else (3, cp, n), rows=rows)
    for name, last in (("pstring_split_once", False), ("pstring_rsplit_once", True)):
        rows = []
        for s in hays:
            for p in pats:
                w = rs_split_once(s, p, last)
                rows.append((S(s, 3) + S(p, cp), [1] + S(w[0], 3) + S(w[1], 3) if w else [0] + S(b"", 3) + S(b"", 3)))
        yield Case(name, name, (3, cp), rows=rows)


def all_cases(name):
    prm = N.classic_params(name)
    m, c = prm["msg_mod"], prm["carry_mod"]
    rng = np.random.default_rng(sum(map(ord, name)))
    yield from integer_cases(m, c, rng)
    yield from shortint_and_bool_cases(m, c, rng)
    yield from string_cases(m, c)
    yield from padded_cases(m, c)


def run_set(name):
    """-> (refused keys, wrong results as (key, args, clear, inputs, want, got))"""
    prm = N.classic_params(name)
    T = prm["msg_mod"] * prm["carry_mod"]
    refused, wrong = set(), []
    for case in all_cases(name):
        try:
            P = Program(case.op, case.args, clear=case.clear, params=prm)
        except NativeError:
            refused.add(case.key)
            continue
        rows = case.expect(P) if case.expect else case.rows
        got = simulate_batch(P.ir(), [r[0] for r in rows], T)
        for (ins, want), g in zip(rows, got):
            if len(want) != len(g) or any(int(a) != int(b) for a, b in zip(want, g)):
                wrong.append((case.key, case.args, case.clear, list(ins), list(want), [int(v) for v in g]))
                break
    return refused, wrong


def compress(keys):
    """{'radix_default_lt@3', '@4', '@5', 'x'} -> ['radix_default_lt@3..5', 'x']: degrees as ranges"""
    plain, deg = set(), {}
    for k in keys:
        if "@" in k:
            op, d = k.split("@")
            deg.setdefault(op, []).append(int(d))
        else:
            plain.add(k)
    out = sorted(plain)
    for op, ds in sorted(deg.items()):
        ds.sort()
        start = prev = ds[0]
        for d in ds[1:] + [None]:
            if d is not None and d == prev + 1:
                prev = d
                continue
            out.append(f"{op}@{start}" if start == prev else f"{op}@{start}..{prev}")
            if d is not None:
                start = prev = d
    return sorted(out)


# ---- which ops each set refuses ------------------------------------------------------------------------------------------------
# The fused case conversion, find / rfind and the null-padded model are written for 2-bit blocks (message modulus 4).
TWO_BIT = frozenset({
    "pstring_concat", "pstring_contains", "pstring_ends_with", "pstring_eq", "pstring_find", "pstring_ge", "pstring_gt",
    "pstring_is_empty", "pstring_le", "pstring_len", "pstring_lt", "pstring_ne", "pstring_repeat", "pstring_replace",
    "pstring_replacen", "pstring_rfind", "pstring_rsplit_once", "pstring_split", "pstring_split_once", "pstring_splitn",
    "pstring_starts_with", "pstring_strip_prefix", "pstring_strip_suffix", "pstring_trim", "pstring_trim_end", "pstring_trim_start",
    "string_eq_ignore_case", "string_eq_ignore_case_packed", "string_find", "string_find/clear", "string_find_packed",
    "string_find_windows", "string_rfind", "string_rfind/clear", "string_rfind_packed", "string_to_lowercase", "string_to_uppercase",
})
# One bivariate PBS packs two blocks as x * msg_mod + y: it needs carry_mod >= msg_mod.  (The packed equalities fall back to it.)
BIVARIATE = frozenset({
    "radix_eq", "radix_eq_packed", "radix_if_then_else", "radix_ne", "radix_scalar_eq", "radix_scalar_gt", "radix_scalar_gt/above",
    "radix_scalar_lt", "radix_scalar_lt/above", "shortint_bivariate_lut", "string_contains", "string_contains/clear",
    "string_contains_many", "string_contains_many_packed", "string_contains_packed", "string_contains_windows", "string_ends_with",
    "string_ends_with/clear", "string_ends_with_packed", "string_eq", "string_eq/clear", "string_eq_many", "string_eq_many_packed",
    "string_eq_packed", "string_ne", "string_ne/clear", "string_ne_many", "string_ne_many_packed", "string_ne_packed",
    "string_starts_with", "string_starts_with/clear", "string_starts_with_packed",
})
# The comparator reduces sign pairs 4 * hi + lo <= 10: it needs a message space of at least 11 values.
COMPARATOR = frozenset({
    "radix_ge", "radix_gt", "radix_le", "radix_lt", "signs_finish", "string_cmp_sign", "string_ge", "string_ge/clear",
    "string_ge_packed", "string_gt", "string_gt/clear", "string_gt_packed", "string_le", "string_le/clear", "string_le_many",
    "string_le_many_packed", "string_le_packed", "string_lt", "string_lt/clear", "string_lt_many", "string_lt_many_packed",
    "string_lt_packed",
})
# Beyond these three groups: carry propagation on one-bit blocks packs a pair of carry states as cur * 3 + prev and needs a message
# space of at least 9 values; the default comparisons refuse when their operands need a propagation that is refused; the boolean
# count trees need at least 3 values; find_combine needs carry_mod >= 2.
REFUSED = {
    "1_0": (TWO_BIT, BIVARIATE, COMPARATOR, "bool_all_true", "bool_any_true", "find_combine", "radix_add", "radix_default_eq@1",
            "radix_default_ge@1", "radix_default_gt@1", "radix_default_le@1", "radix_default_lt@1", "radix_default_ne@1",
            "radix_full_propagate@1"),
    "1_1": (TWO_BIT, COMPARATOR, "radix_add", "radix_default_eq@2..3", "radix_default_ge@1..3", "radix_default_gt@1..3",
            "radix_default_le@1..3", "radix_default_lt@1..3", "radix_default_ne@2..3", "radix_full_propagate@1..3", "radix_scalar_gt",
            "radix_scalar_gt/above", "radix_scalar_lt", "radix_scalar_lt/above"),
    "2_0": (TWO_BIT, BIVARIATE, COMPARATOR, "find_combine", "radix_add", "radix_default_eq@3", "radix_default_ge@3",
            "radix_default_gt@3", "radix_default_le@3", "radix_default_lt@3", "radix_default_ne@3", "radix_full_propagate@3"),
    "1_2": (TWO_BIT, COMPARATOR, "radix_add", "radix_default_eq@2..7", "radix_default_ge@1..7", "radix_default_gt@1..7",
            "radix_default_le@1..7", "radix_default_lt@1..7", "radix_default_ne@2..7", "radix_full_propagate@1..7", "radix_scalar_gt",
            "radix_scalar_gt/above", "radix_scalar_lt", "radix_scalar_lt/above"),
    "2_1": (TWO_BIT, BIVARIATE, COMPARATOR, "radix_add", "radix_default_eq@3..7", "radix_default_ge@3..7", "radix_default_gt@3..7",
            "radix_default_le@3..7", "radix_default_lt@3..7", "radix_default_ne@3..7", "radix_full_propagate@3..7"),
    "3_0": (TWO_BIT, BIVARIATE, COMPARATOR, "find_combine", "radix_add", "radix_default_eq@7", "radix_default_ge@7",
            "radix_default_gt@7", "radix_default_le@7", "radix_default_lt@7", "radix_default_ne@7", "radix_full_propagate@7"),
    "1_3": (TWO_BIT,),
    "2_2": (),
    "3_1": (TWO_BIT, BIVARIATE, "radix_add", "radix_default_eq@7..15", "radix_default_ge@8..15", "radix_default_gt@8..15",
            "radix_default_le@8..15", "radix_default_lt@8..15", "radix_default_ne@7..15", "radix_full_propagate@7..15"),
    "4_0": (TWO_BIT, BIVARIATE, "find_combine", "radix_add", "radix_default_eq@15", "radix_default_ne@15", "radix_full_propagate@15"),
    "1_4": (TWO_BIT,),
    "2_3": (),
    "3_2": (TWO_BIT, BIVARIATE, "radix_add", "radix_default_eq@7..31", "radix_default_ge@8..31", "radix_default_gt@8..31",
            "radix_default_le@8..31", "radix_default_lt@8..31", "radix_default_ne@7..31", "radix_full_propagate@7..31"),
    "4_1": (TWO_BIT, BIVARIATE, "radix_add", "radix_default_eq@15..31", "radix_default_ge@16..31", "radix_default_gt@16..31",
            "radix_default_le@16..31", "radix_default_lt@16..31", "radix_default_ne@15..31", "radix_full_propagate@15..31"),
    "5_0": (TWO_BIT, BIVARIATE, "find_combine", "radix_add", "radix_default_eq@31", "radix_default_ne@31", "radix_full_propagate@31"),
    "1_5": (TWO_BIT,),
    "2_4": (),
    "3_3": (TWO_BIT,),
    "4_2": (TWO_BIT, BIVARIATE, "radix_add", "radix_default_eq@15..63", "radix_default_ge@16..63", "radix_default_gt@16..63",
            "radix_default_le@16..63", "radix_default_lt@16..63", "radix_default_ne@15..63", "radix_full_propagate@15..63"),
    "5_1": (TWO_BIT, BIVARIATE, "radix_add", "radix_default_eq@31..63", "radix_default_ge@32..63", "radix_default_gt@32..63",
            "radix_default_le@32..63", "radix_default_lt@32..63", "radix_default_ne@31..63", "radix_full_propagate@31..63"),
    "6_0": (TWO_BIT, BIVARIATE, "find_combine", "radix_add", "radix_default_eq@63", "radix_default_ne@63", "radix_full_propagate@63"),
    "1_6": (TWO_BIT,),
    "2_5": (),
    "3_4": (TWO_BIT,),
    "4_3": (TWO_BIT, BIVARIATE, "radix_add", "radix_default_eq@15..127", "radix_default_ge@16..127", "radix_default_gt@16..127",
            "radix_default_le@16..127", "radix_default_lt@16..127", "radix_default_ne@15..127", "radix_full_propagate@15..127"),
    "5_2": (TWO_BIT, BIVARIATE, "radix_add", "radix_default_eq@31..127", "radix_default_ge@32..127", "radix_default_gt@32..127",
            "radix_default_le@32..127", "radix_default_lt@32..127", "radix_default_ne@31..127", "radix_full_propagate@31..127"),
    "6_1": (TWO_BIT, BIVARIATE, "radix_add", "radix_default_eq@63..127", "radix_default_ge@64..127", "radix_default_gt@64..127",
            "radix_default_le@64..127", "radix_default_lt@64..127", "radix_default_ne@63..127", "radix_full_propagate@63..127"),
    "7_0": (TWO_BIT, BIVARIATE, "find_combine", "radix_add", "radix_default_eq@127", "radix_default_ne@127",
            "radix_full_propagate@127"),
    "1_7": (TWO_BIT,),
    "2_6": (),
    "3_5": (TWO_BIT,),
    "4_4": (TWO_BIT,),
    "5_3": (TWO_BIT, BIVARIATE, "radix_add", "radix_default_eq@31..255", "radix_default_ge@32..255", "radix_default_gt@32..255",
            "radix_default_le@32..255", "radix_default_lt@32..255", "radix_default_ne@31..255", "radix_full_propagate@31..255"),
    "6_2": (TWO_BIT, BIVARIATE, "radix_add", "radix_default_eq@63..255", "radix_default_ge@64..255", "radix_default_gt@64..255",
            "radix_default_le@64..255", "radix_default_lt@64..255", "radix_default_ne@63..255", "radix_full_propagate@63..255"),
    "7_1": (TWO_BIT, BIVARIATE, "radix_add", "radix_default_eq@127..255", "radix_default_ge@128..255", "radix_default_gt@128..255",
            "radix_default_le@128..255", "radix_default_lt@128..255", "radix_default_ne@127..255", "radix_full_propagate@127..255"),
    "8_0": (TWO_BIT, BIVARIATE, "find_combine", "radix_add", "radix_default_eq@255", "radix_default_ne@255",
            "radix_full_propagate@255"),
}


def expand(entry):
    out = set()
    for item in entry:
        out |= set(item) if isinstance(item, frozenset) else {item}
    return sorted(out)


def test_refusal_table_is_consistent():
    assert set(REFUSED) == set(SETS) and len(SETS) == 36
    two_bit = [s for s in SETS if N.classic_params(s)["msg_mod"] != 4]
    assert all(TWO_BIT <= set(expand(REFUSED[s])) for s in two_bit)
    assert [s for s in SETS if not REFUSED[s]] == ["2_2", "2_3", "2_4", "2_5", "2_6"]     # msg_mod 4 with carry_mod >= 4: everything


@pytest.mark.parametrize("name", SETS)
def test_every_op_at_every_modulus(name):
    """every op of the program API on this set's moduli: the right value on every input row, or NativeError; the refusals as pinned"""
    refused, wrong = run_set(name)
    assert not wrong, f"{name}: {len(wrong)} ops return a wrong value, first: {wrong[:3]}"
    assert compress(refused) == expand(REFUSED[name])


def test_compress_ranges():
    assert compress({"a@3", "a@4", "a@5", "a@7", "b", "c@1"}) == ["a@3..5", "a@7", "b", "c@1"]


def test_clear_operand_with_nul_is_refused():
    """the C ABI takes the clear operand as a NUL-terminated string: a NUL char would silently cut the pattern short"""
    with pytest.raises(ValueError, match="NUL"):
        Program("string_eq", (2,), clear="\x00\x01")
    with pytest.raises(ValueError, match="NUL"):
        Program("pstring_strip_prefix", (4,), clear=b"a\x00")


def test_propagation_shapes():
    """degree 2m - 1 takes the extraction (it used to go straight to single-carry propagation); degrees that allow a single carry
    keep the programs test_host_programs.py pins; carry_mod > msg_mod can take more than one extraction"""
    assert Program("radix_full_propagate", (3, 6)).n_pbs == Program("radix_add", (3,)).n_pbs
    assert Program("radix_full_propagate", (3, 7)).n_pbs == Program("radix_full_propagate", (3, 15)).n_pbs
    assert Program("radix_full_propagate", (3, 7)).n_levels == Program("radix_full_propagate", (3, 6)).n_levels + 1
    p23 = N.classic_params("2_3")                       # m 4, c 8: 31 -> 3 + 7 = 10 > 6 -> 3 + 2 = 5
    assert Program("radix_full_propagate", (3, 31), params=p23).n_levels == Program("radix_full_propagate", (3, 7), params=p23).n_levels + 1


# ---- the findings with real KS-PBS on the toy keys -----------------------------------------------------------------------------
def _toy(orc, msg_mod, carry_mod):
    p = orc.params("toy")
    p.msg_mod, p.carry_mod = msg_mod, carry_mod
    p.poly_size = max(256, 16 * msg_mod * carry_mod)    # a box of the lookup table must stay wider than the modulus-switch rounding
    ck = orc.ClientKey(p, 0xA110 + msg_mod * carry_mod)
    sk = orc.ServerKey(ck, 0xA120 + msg_mod * carry_mod)
    return p, ck, sk


def _run_real(orc, keys, op, args, blocks, clear=None):
    from oracle import radix as R
    p, ck, sk = keys
    P = Program(op, args, clear=clear, params=engine_params(p))
    ins = np.stack([ck.encrypt_with_carry(int(b)) for b in blocks])
    return [ck.decrypt_message_and_carry(c) for c in R.run_program(P.ir(), sk, ins)]


def test_degree_2m_minus_1_propagates_real_pbs(orc):
    """2_2 moduli: blocks [7, 7, 7] hold 7 + 28 + 112 = 147 = 19 mod 64 = [3, 0, 1]; a block of 7 plus a carry is 8, two carries out"""
    keys = _toy(orc, 4, 4)
    assert _run_real(orc, keys, "radix_full_propagate", (3, 7), [7, 7, 7]) == [3, 0, 1]
    assert _run_real(orc, keys, "radix_default_eq", (3, 7), [7, 7, 7, 3, 0, 1]) == [1]
    assert _run_real(orc, keys, "radix_default_lt", (3, 7), [7, 7, 7, 0, 1, 1]) == [1]       # 19 < 20


def test_carry_mod_above_msg_mod_propagates_real_pbs(orc):
    """2_3 moduli (m 4, c 8): [31, 31, 31] = 651 = 11 mod 64 = [3, 2, 0]: one extraction leaves 3 + 7 = 10 > 2m - 2, so it repeats"""
    keys = _toy(orc, 4, 8)
    assert _run_real(orc, keys, "radix_full_propagate", (3, 31), [31, 31, 31]) == [3, 2, 0]


def test_one_bit_blocks_add_real_pbs(orc):
    """1_3 moduli (m 2, c 8): the carry states {0, 1, 2} need an injective packing; 7 + 1 = 8 = 0 mod 8, 31 + 0 = 31"""
    keys = _toy(orc, 2, 8)
    assert _run_real(orc, keys, "radix_add", (3,), [1, 1, 1, 1, 0, 0]) == [0, 0, 0]
    assert _run_real(orc, keys, "radix_add", (5,), [1] * 5 + [0] * 5) == [1] * 5
    assert _run_real(orc, keys, "radix_full_propagate", (5, 2), [2, 1, 1, 1, 1]) == [0, 0, 0, 0, 0]    # 2 + 30 = 32 = 0 mod 32


def test_packed_equality_with_small_carry(orc):
    """hi * m + lo fits the message space only when carry_mod >= msg_mod.  3_0 and 3_1 used to report "zz~".ends_with("zz") and 8_0
    returned 511 for an equality; they now refuse (the per-block fallback needs the same carry space).  The same pairs on 3_3 moduli
    (m 8, c 8), where the packed path is valid, with real KS-PBS."""
    for name in ("3_0", "3_1", "8_0"):
        for op, args in (("string_ends_with_packed", (3, 2)), ("string_eq_packed", (2, 2))):
            with pytest.raises(NativeError, match="degree"):
                Program(op, args, params=N.classic_params(name))
    keys = _toy(orc, 8, 8)
    s = lambda x: str_blocks(x, 8)
    assert _run_real(orc, keys, "string_ends_with_packed", (3, 2), s(b"zz~") + s(b"zz")) == [0]
    assert _run_real(orc, keys, "string_ends_with_packed", (3, 2), s(b"~zz") + s(b"zz")) == [1]
    assert _run_real(orc, keys, "string_eq_packed", (2, 2), s(b"\x7f\x00") + s(b"\x7f\x01")) == [0]
