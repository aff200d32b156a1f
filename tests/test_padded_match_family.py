"""Null-padded matches / match_indices / rmatch_indices / trim_start_matches / trim_end_matches / lines / split_whitespace
(host/padded.h) on CPU.

The recorded programs are executed noise-free on plaintexts, many input rows at once, against a reference of Rust's str semantics
pinned against Python where the two agree.  Every string up to capacity 5 over {a, b, \\n, \\r, ' '} is tried; split_whitespace also
gets every multi-byte Unicode whitespace sequence and their near misses.  The noise and depth bounds are read from the program IR,
and a few small cases run through the CPU oracle's real KS-PBS on the toy keys."""
import itertools
import random

import numpy as np
import pytest

from fhe_string_bounty_b200 import NativeError, _native as N
from fhe_string_bounty_b200.host import Program
from helpers import engine_params, string_blocks_clear
from test_padded_split_family import build, check_split_rows, rs_rmatches, rs_split_inclusive, simulate_rows, to_bytes, to_int
from test_padded_split_replace import digits_for, max_matches, pad, rs_matches

# char::is_whitespace: Unicode White_Space (Python's str.isspace() adds U+001C ..= U+001F)
WS_CHARS = [chr(c) for c in (*range(0x09, 0x0E), 0x20, 0x85, 0xA0, 0x1680, *range(0x2000, 0x200B), 0x2028, 0x2029, 0x202F, 0x205F, 0x3000)]
WS_SEQS = sorted({c.encode() for c in WS_CHARS}, key=lambda b: (len(b), b))


# ---- reference: Rust's str methods -----------------------------------------------------------------------------------------------------
def rs_match_indices(s, pat):
    return rs_matches(s, pat)


def rs_rmatch_indices(s, pat):
    return rs_rmatches(s, pat)


def rs_trim_start_matches(s, pat):
    if pat:
        while s.startswith(pat):
            s = s[len(pat):]
    return s


def rs_trim_end_matches(s, pat):
    if pat:
        while s.endswith(pat):
            s = s[:len(s) - len(pat)]
    return s


def rs_lines(s):
    out = []
    for line in rs_split_inclusive(s, b"\n"):
        if line.endswith(b"\n"):
            line = line[:-1]
            if line.endswith(b"\r"):
                line = line[:-1]
        out.append(line)
    return out


def rs_split_whitespace(s):
    """every occurrence of a White_Space UTF-8 sequence separates; the rest are word bytes"""
    out, cur, i = [], b"", 0
    while i < len(s):
        seq = next((w for w in WS_SEQS if s.startswith(w, i)), None)
        if seq is None:
            cur += s[i:i + 1]
            i += 1
            continue
        if cur:
            out.append(cur)
        cur = b""
        i += len(seq)
    return out + ([cur] if cur else [])


def test_reference_against_python():
    assert len(WS_CHARS) == 25 and [len(b) for b in WS_SEQS].count(1) == 6 and [len(b) for b in WS_SEQS].count(2) == 2
    assert {chr(c) for c in range(0x110000) if chr(c).isspace()} - {"\x1c", "\x1d", "\x1e", "\x1f"} == set(WS_CHARS)
    words = [b"", b"a", b"aa", b"aaa", b"aaaaa", b"ababa", b"babab", b"abcab", b"a,b,,c", b"xyz", b", x, ", b"abab", b"xabab"]
    pats = [b"a", b"aa", b"ab", b"aba", b"bab", b",", b", ", b"x", b"zz"]
    for s in words:
        for p in pats:
            want, i = [], 0
            while (j := s.find(p, i)) >= 0:
                want.append(j)
                i = j + len(p)
            assert rs_match_indices(s, p) == want and s.count(p) == len(want)
            want, end = [], len(s)
            while (j := s.rfind(p, 0, end)) >= 0:
                want.append(j)
                end = j
            assert rs_rmatch_indices(s, p) == want
            assert len(rs_rmatch_indices(s, p)) == len(rs_match_indices(s, p))      # no separate rmatches count
            if len(p) == 1:
                assert rs_trim_start_matches(s, p) == s.lstrip(p) and rs_trim_end_matches(s, p) == s.rstrip(p)
        assert len(rs_rmatch_indices(s, b"")) == len(rs_match_indices(s, b"")) == len(s) + 1
    for t in ("a b", "  a\t\tb\n c \r\x0c", "x\xa0y\u2003z\u3000", "\u1680\u202f\u205f", "\xe9 \xfc\x85\xf1", "", " ", "\u200bx", "a\u2028b\u2029"):
        assert rs_split_whitespace(t.encode()) == [w.encode() for w in t.split()], t
    for t in ("a\nb", "a\r\nb\n", "x\n\ny", "\n", "a"):
        assert rs_lines(t.encode()) == [w.encode() for w in t.splitlines()], t
    # Rust only (std's doc examples and the cases Python does not share)
    assert rs_match_indices(b"ababa", b"aba") == [0] and rs_rmatch_indices(b"ababa", b"aba") == [2]
    assert rs_match_indices(b"ab", b"") == [0, 1, 2] and rs_rmatch_indices(b"ab", b"") == [2, 1, 0]
    assert rs_trim_start_matches(b"aaa", b"aa") == b"a" and rs_trim_end_matches(b"aaa", b"aa") == b"a"
    assert rs_trim_start_matches(b"ababx", b"ab") == b"x" and rs_trim_end_matches(b"xabab", b"ab") == b"x"
    assert rs_trim_start_matches(b"ab", b"") == b"ab" and rs_trim_end_matches(b"ab", b"") == b"ab"
    assert rs_lines(b"foo\nbar\n\r\nbaz\r") == [b"foo", b"bar", b"", b"baz\r"]
    assert rs_lines(b"a\n") == [b"a"] and rs_lines(b"\n") == [b""] and rs_lines(b"") == [] and rs_lines(b"\r\r\n") == [b"\r"]
    assert rs_split_whitespace(b"a\x0bb c") == [b"a", b"b", b"c"] and rs_split_whitespace(b"a\x1cb") == [b"a\x1cb"]


# ---- noise-free execution ----------------------------------------------------------------------------------------------------------------
CAP = 5
ALPHABET = b"ab\n\r "
ALL = [bytes(t) for k in range(CAP + 1) for t in itertools.product(ALPHABET, repeat=k)]      # 3906 strings
PADDED = [b"", b"a", b"aa", b"aba"]                           # each at every capacity from its length to 3
CLEAR = ["a", "aa", "ab", "aba", "bab", "\n", "\r\n"]        # self-overlapping "aa", "aba", "bab"


def pattern_specs():
    for cp in range(4):
        yield f"padded{cp}", [p for p in PADDED if len(p) <= cp], cp, None
    for c in CLEAR:
        yield f"clear-{c.encode().hex()}", [c.encode()], len(c), c


SPECS = list(pattern_specs())
IDS = [s[0] for s in SPECS]


def run_rows(op, args, clear, rows, chunk=1500):
    prog, ir = build(op, args, clear)
    out = np.concatenate([simulate_rows(ir, rows[i:i + chunk]) for i in range(0, len(rows), chunk)]) if rows else np.zeros((0, prog.n_outputs))
    return prog, out


def pattern_rows(pats, cp, clear):
    cases = [(s, p) for s in ALL for p in pats]
    return cases, [string_blocks_clear(pad(s, CAP)) + ([] if clear else string_blocks_clear(pad(p, cp))) for s, p in cases]


@pytest.mark.parametrize("spec", SPECS, ids=IDS)
def test_matches_clear_simulation(spec):
    """matches, match_indices and rmatch_indices: count (digits_for(M)) then M indices of digits_for(capacity) digits, zero past the count"""
    _, pats, cp, clear = spec
    M = max_matches(CAP, cp if clear else 0)
    nd, ni = digits_for(M), digits_for(CAP)
    cases, rows = pattern_rows(pats, cp, clear)
    prog, out = run_rows("pstring_matches", (CAP, cp), clear, rows)
    assert prog.n_outputs == nd
    for (s, p), o in zip(cases, out):
        assert to_int(o) == len(rs_match_indices(s, p)), (s, p, clear)
    for op, ref in (("pstring_match_indices", rs_match_indices), ("pstring_rmatch_indices", rs_rmatch_indices)):
        prog, out = run_rows(op, (CAP, cp), clear, rows)
        assert prog.n_outputs == nd + M * ni
        for (s, p), o in zip(cases, out):
            want = ref(s, p)
            got = [to_int(o[nd + ni * k: nd + ni * (k + 1)]) for k in range(M)]
            assert (to_int(o[:nd]), got) == (len(want), want + [0] * (M - len(want))), (op, s, p, clear)


@pytest.mark.parametrize("spec", SPECS, ids=IDS)
def test_trim_matches_clear_simulation(spec):
    _, pats, cp, clear = spec
    cases, rows = pattern_rows(pats, cp, clear)
    for op, ref in (("pstring_trim_start_matches", rs_trim_start_matches), ("pstring_trim_end_matches", rs_trim_end_matches)):
        prog, out = run_rows(op, (CAP, cp), clear, rows)
        assert prog.n_outputs == 4 * CAP
        for (s, p), o in zip(cases, out):
            assert to_bytes(o) == pad(ref(s, p), CAP), (op, s, p, clear)


def test_lines_clear_simulation():
    for cap in (0, 1, 3, CAP):
        check_split_rows("pstring_lines", (cap,), None, cap, cap, [(s, None, rs_lines(s), []) for s in ALL if len(s) <= cap])
    # the count has digits_for(capacity) blocks (one fewer than split_inclusive's at capacity 4 ** k - 1)
    check_split_rows("pstring_lines", (3,), None, 3, 3, [(b"\n\n\n", None, [b"", b"", b""], []), (b"a\nb", None, [b"a", b"b"], [])])


def whitespace_cases():
    """every White_Space sequence at the start, in the middle and at the end, alone and twice; near misses that are not whitespace"""
    cases = [s for s in ALL]
    for w in WS_SEQS:
        cases += [w, w + b"ab", b"x" + w + b"y", b"ab" + w, w + w, b"a" + w + b"\n" + w]
    near = [b"\xe2\x80\x8b", b"\xe2\x80\xb0", b"\xe2\x80\xa7", b"\xe2\x80\xaa", b"\xe2\x81\x9e", b"\xe2\x81\xa0", b"\xe1\x9a\x81",
            b"\xe1\x9b\x80", b"\xe3\x80\x81", b"\xe3\x81\x80", b"\xc2\x80", b"\xc2\x84", b"\xc2\xa1", b"\xc3\x85", b"\xc2", b"\xe2\x80",
            b"\x85", b"\xa0", b"\x80\x80", b"\x1c", b"\x1f", b"\x08", b"\x0e", b"\xe2\x82\x80", b"\xe2\x80\x8f", b"\xe2\x80\xaf\xaf"]
    for w in near:
        cases += [w, b"a" + w + b" b", b" " + w]
    cases += [b"\xe2\xe2\x80\x80\x80", b"\xc2\xc2\x85\x85", b"\xe1\xe1\x9a\x80", b"\xe3\x80\xe3\x80\x80"]
    rnd = random.Random(0x5EED)
    pool = [0x09, 0x0B, 0x20, 0x61, 0xC2, 0xE1, 0xE2, 0xE3, 0x80, 0x81, 0x85, 0x8A, 0x8B, 0x9A, 0x9F, 0xA0, 0xA8, 0xA9, 0xAF, 0xB0]
    cases += [bytes(rnd.choice(pool) for _ in range(rnd.randint(1, 9))) for _ in range(3000)]
    return cases


def test_split_whitespace_clear_simulation():
    cap = 9
    cases = [s for s in whitespace_cases() if len(s) <= cap]
    check_split_rows("pstring_split_whitespace", (cap,), None, cap, (cap + 1) // 2, [(s, None, rs_split_whitespace(s), []) for s in cases])
    for cap in (0, 1, 2):
        check_split_rows("pstring_split_whitespace", (cap,), None, cap, (cap + 1) // 2,
                         [(s, None, rs_split_whitespace(s), []) for s in ALL if len(s) <= cap])


def test_split_whitespace_cost():
    """the byte classification costs 18 PBS per byte where split_ascii_whitespace spends 3; the rest is the same split"""
    for cap in (6, 16):
        a, u = Program("pstring_split_ascii_whitespace", (cap,)), Program("pstring_split_whitespace", (cap,))
        assert u.n_outputs == a.n_outputs
        assert u.n_pbs - a.n_pbs <= 15 * cap, (cap, u.n_pbs, a.n_pbs)


def test_shapes():
    # the documented output counts, empty capacities included
    assert Program("pstring_matches", (0, 0)).n_outputs == digits_for(1)
    assert Program("pstring_matches", (4, 5), clear="abcde").n_outputs == 1
    assert Program("pstring_match_indices", (4, 5), clear="abcde").n_outputs == 1                 # M = 0: the count only
    assert Program("pstring_rmatch_indices", (6, 2)).n_outputs == digits_for(7) + 7 * digits_for(6)
    assert Program("pstring_match_indices", (16, 2), clear="ab").n_outputs == digits_for(8) + 8 * digits_for(16)
    assert Program("pstring_trim_start_matches", (6, 0)).n_outputs == 24 and Program("pstring_trim_end_matches", (0, 2)).n_outputs == 0
    assert Program("pstring_lines", (0,)).n_outputs == 1 and Program("pstring_lines", (4,)).n_outputs == digits_for(4) + 4 * 4 * 4
    assert Program("pstring_split_whitespace", (7,)).n_outputs == digits_for(4) + 4 * 7 * 4
    assert Program("pstring_trim_end_matches", (6, 2), clear="ab").n_inputs == 24 and Program("pstring_matches", (6, 2)).n_inputs == 32
    # a padded pattern selects among the candidate lengths: no chain as long as the string, for trim_* with any pattern
    for op in ("pstring_trim_start_matches", "pstring_trim_end_matches"):
        assert Program(op, (64, 4)).n_levels < 48 and Program(op, (64, 2), clear="ab").n_levels < 24, op
    assert Program("pstring_match_indices", (64, 2), clear="ab").n_levels < 64 and Program("pstring_lines", (32,)).n_levels < 32
    # larger programs keep the noise bound and the result-block invariant
    for op, args, clear in (("pstring_matches", (12, 4), None), ("pstring_match_indices", (12, 3), "aba"), ("pstring_rmatch_indices", (12, 4), None),
                            ("pstring_trim_start_matches", (12, 5), None), ("pstring_trim_end_matches", (12, 5), None),
                            ("pstring_trim_end_matches", (12, 3), "aba"), ("pstring_lines", (16,), None), ("pstring_split_whitespace", (16,), None)):
        build(op, args, clear)


NEW_OPS = [("pstring_matches", (6, 2)), ("pstring_match_indices", (6, 2)), ("pstring_rmatch_indices", (6, 2)),
           ("pstring_trim_start_matches", (6, 2)), ("pstring_trim_end_matches", (6, 2)), ("pstring_lines", (6,)),
           ("pstring_split_whitespace", (6,))]


def test_argument_errors():
    for op, args in NEW_OPS:
        with pytest.raises(NativeError, match="expected"):
            Program(op, args[:-1])
    for op, _ in NEW_OPS[:5]:
        with pytest.raises(NativeError, match="differs from the clear pattern's length"):
            Program(op, (8, 3), clear="ab")
    for op in ("pstring_lines", "pstring_split_whitespace"):
        with pytest.raises(NativeError, match="no clear operand"):
            Program(op, (6,), clear="ab")
    for op, args in (("pstring_matches", (2**21, 1)), ("pstring_match_indices", (8, 2**21)), ("pstring_trim_end_matches", (2**40, 2)),
                     ("pstring_trim_start_matches", (2**20 + 1, 0)), ("pstring_lines", (2**21,)), ("pstring_split_whitespace", (2**60,))):
        with pytest.raises(NativeError, match="limited"):
            Program(op, args)
    for op, args in (("pstring_lines", (2**10 + 1,)), ("pstring_split_whitespace", (2**11,)), ("pstring_match_indices", (2**10, 0)),
                     ("pstring_rmatch_indices", (2**11, 1))):
        with pytest.raises(NativeError, match="exceed"):
            Program(op, args)


def test_other_moduli_refused():
    """every new op refuses the 36 classic sets whose message modulus is not 4, and builds on 2_2 ... 2_6"""
    sets = list(N._CLASSIC_SETS)
    assert len(sets) == 36
    for name in sets:
        prm = N.classic_params(name)
        for op, args in NEW_OPS:
            if prm["msg_mod"] != 4:
                with pytest.raises(NativeError, match="message modulus 4"):
                    Program(op, args, params=prm)
            elif name in ("2_2", "2_3", "2_4", "2_5", "2_6"):
                assert Program(op, args, params=prm).n_pbs > 0, (name, op)


def test_match_family_with_real_pbs_toy(orc, toy_keys):
    """small programs executed with the oracle's CPU KS-PBS on the toy parameter set"""
    from oracle import radix as R
    p, ck, sk = toy_keys
    prm = engine_params(p)
    enc = lambda *xs: np.concatenate([R.encrypt_string(ck, pad(x, c)) for x, c in xs])
    out = R.run_program(Program("pstring_rmatch_indices", (4, 2), params=prm).ir(), sk, enc((b"abab", 4), (b"ab", 2)))
    nd, ni = digits_for(5), digits_for(4)
    assert R.decrypt_radix(ck, out[:nd]) == 2
    assert [R.decrypt_radix(ck, out[nd + ni * k: nd + ni * (k + 1)]) for k in range(5)] == [2, 0, 0, 0, 0]
    out = R.run_program(Program("pstring_trim_end_matches", (4, 1), clear="a", params=prm).ir(), sk, enc((b"baa", 4)))
    assert R.decrypt_string(ck, out) == pad(b"b", 4)
    out = R.run_program(Program("pstring_lines", (3,), params=prm).ir(), sk, enc((b"a\r\n", 3)))
    nd = digits_for(3)
    assert R.decrypt_radix(ck, out[:nd]) == 1 and R.decrypt_string(ck, out[nd:nd + 12]) == pad(b"a", 3)
