"""Null-padded rsplit / rsplitn / split_terminator / rsplit_terminator / split_inclusive / split_ascii_whitespace, the ops with a secret
integer argument (repeat_enc, replacen_enc, splitn_enc, rsplitn_enc), strip_prefix / strip_suffix with a padded pattern and the padded
eq_ignore_case (host/padded.h) on CPU.

The recorded programs are executed noise-free on plaintexts, many input rows at once, against a reference of Rust's str semantics pinned
against Python's bytes methods where the two agree.  The noise and depth bounds are read from the program IR, and three small cases run
through the CPU oracle's real KS-PBS on the toy keys."""
import numpy as np
import pytest

from fhe_string_bounty_b200 import NativeError, _native as N
from fhe_string_bounty_b200.host import Program
from helpers import engine_params, string_blocks_clear
from test_padded_split_replace import digits_for, max_matches, pad, pbs_input_noise, rs_matches, rs_replacen, rs_splitn, well_formed

ASCII_WS = b"\t\n\x0c\r "          # u8::is_ascii_whitespace (no U+000B)


# ---- reference: Rust's str methods with a &str pattern ------------------------------------------------------------------------------
def rs_rmatches(s, pat):
    """reverse searcher: rightmost non-overlapping, right to left"""
    if not pat:
        return list(range(len(s), -1, -1))
    out, end = [], len(s)
    while (j := s.rfind(pat, 0, end)) >= 0:
        out.append(j)
        end = j
    return out


def rs_rsplitn(s, pat, n=None):
    if n == 0:
        return []
    ms = rs_rmatches(s, pat)[:None if n is None else n - 1]
    parts, end = [], len(s)
    for m in ms:
        parts.append(s[m + len(pat):end])
        end = m
    return parts + [s[:end]]


def rs_split_terminator(s, pat):
    parts = rs_splitn(s, pat)
    return parts[:-1] if parts[-1] == b"" else parts


def rs_rsplit_terminator(s, pat):
    parts = rs_rsplitn(s, pat)
    return parts[1:] if parts[0] == b"" else parts


def rs_split_inclusive(s, pat):
    parts, start = [], 0
    for m in rs_matches(s, pat):
        parts.append(s[start:m + len(pat)])
        start = m + len(pat)
    return parts + ([s[start:]] if start < len(s) else [])


def rs_split_ascii_whitespace(s):
    out, cur = [], b""
    for ch in s:
        if ch in ASCII_WS:
            if cur:
                out.append(cur)
            cur = b""
        else:
            cur += bytes([ch])
    return out + ([cur] if cur else [])


def test_reference_against_python():
    words = [b"", b"a", b"aa", b"aaa", b"aaaaa", b"ababa", b"babab", b"abcab", b"a,b,,c", b"xyz", b", x, ", b"a\nb\n", b"\n\nx"]
    pats = [b"a", b"aa", b"ab", b"aba", b"bab", b",", b", ", b"x", b"zz", b"\n"]
    for s in words:
        for p in pats:
            assert rs_rsplitn(s, p) == s.rsplit(p)[::-1]
            for n in range(1, 5):
                assert rs_rsplitn(s, p, n) == s.rsplit(p, n - 1)[::-1]
            assert rs_rsplitn(s, p, 0) == []
        assert rs_split_inclusive(s, b"\n") == s.splitlines(keepends=True)
    for s in (b"", b" ", b"a b", b"  a\t\tb\n c \r\x0c", b"ab", b"\x00 x"):
        assert rs_split_ascii_whitespace(s) == s.split()
    # Rust only: the empty pattern, the empty string, both terminators, U+000B
    assert rs_rmatches(b"ab", b"") == [2, 1, 0]
    assert rs_rsplitn(b"ab", b"") == [b"", b"b", b"a", b""]
    assert rs_rsplitn(b"babab", b"bab") == [b"", b"ba"] and rs_splitn(b"babab", b"bab") == [b"", b"ab"]
    assert rs_rsplitn(b"ab", b"", 2) == [b"", b"ab"]
    assert rs_split_terminator(b"", b"x") == [] and rs_split_terminator(b"", b"") == [b""]
    assert rs_split_terminator(b"a,b,", b",") == [b"a", b"b"] and rs_split_terminator(b"a,b", b",") == [b"a", b"b"]
    assert rs_split_terminator(b"ab", b"") == [b"", b"a", b"b"]
    assert rs_rsplit_terminator(b"A..B..", b".") == [b"", b"B", b"", b"A"]
    assert rs_rsplit_terminator(b"", b"x") == [] and rs_rsplit_terminator(b"", b"") == [b""]
    assert rs_rsplit_terminator(b"ab", b"") == [b"b", b"a", b""]
    assert rs_split_inclusive(b"a\nb\n", b"\n") == [b"a\n", b"b\n"] and rs_split_inclusive(b"", b"\n") == []
    assert rs_split_inclusive(b"ab", b"") == [b"", b"a", b"b"] and rs_split_inclusive(b"", b"") == [b""]
    assert rs_split_ascii_whitespace(b"a\x0bb c") == [b"a\x0bb", b"c"]


# ---- noise-free execution -------------------------------------------------------------------------------------------------------------
def simulate_rows(ir, rows, total_mod=16):
    """the program on plaintext input rows [batch, n_inputs] -> outputs [batch, n_outputs]; asserts that no PBS operand reaches the
    padding bit (a slot holds its value modulo 2 * total_mod)"""
    T, M = total_mod, 2 * total_mod
    delta = (1 << 63) // T
    rows = np.asarray(rows, dtype=np.int64).reshape(len(rows), ir.n_inputs)
    val = np.zeros((ir.n_slots, rows.shape[0]), dtype=np.int64)
    val[: ir.n_inputs] = rows.T
    tables = ir.lut_tables.astype(np.int64)
    for lv in range(len(ir.level_lin_off) - 1):
        for li in range(int(ir.level_lin_off[lv]), int(ir.level_lin_off[lv + 1])):
            out, tb, te = (int(v) for v in ir.lin[li])
            acc = np.full(rows.shape[0], int(ir.lin_body[li]) // delta, dtype=np.int64)
            for t in range(tb, te):
                acc += int(ir.term_coef[t]) * val[int(ir.term_slot[t])]
            val[out] = acc % M
        p0, p1 = int(ir.level_pbs_off[lv]), int(ir.level_pbs_off[lv + 1])
        if p1 > p0:
            x = val[ir.pbs[p0:p1, 0]]
            assert (x < T).all(), "a PBS operand reached the padding bit"
            val[ir.pbs[p0:p1, 1]] = tables[ir.pbs[p0:p1, 2][:, None], x]
    return val[ir.outputs].T


def build(op, args, clear=None):
    """the program, with the IR checks: no PBS input above 15 nominal noise units, every result block a PBS output or trivial"""
    P = Program(op, args, clear=clear)
    ir = P.ir()
    assert pbs_input_noise(ir) <= 15, (op, args, clear)
    assert int(ir.output_degree_noise[:, 1].max(initial=0)) <= 1 and int(ir.output_degree_noise[:, 0].max(initial=0)) <= 3, (op, args, clear)
    return P, ir


def to_bytes(blocks) -> bytes:
    return bytes(sum(int(d) << (2 * i) for i, d in enumerate(blocks[k:k + 4])) for k in range(0, len(blocks), 4))


def to_int(blocks) -> int:
    return sum(int(d) << (2 * i) for i, d in enumerate(blocks))


def radix(v, nb):
    return [(v >> (2 * i)) & 3 for i in range(nb)]


def split_out(out, nd, cap, P):
    return to_int(out[:nd]), [to_bytes(out[nd + 4 * cap * k: nd + 4 * cap * (k + 1)]) for k in range(P)]


def check_split_rows(op, args, clear, cap, P, cases):
    """cases: [(s, pat, want parts, extra inputs)]: count (digits_for(P) blocks) and P parts of cap chars, parts past the count zero"""
    prog, ir = build(op, args, clear)
    nd = digits_for(P)
    assert prog.n_outputs == nd + 4 * cap * P, (op, args, prog.n_outputs)
    rows = []
    for s, pat, want, ext in cases:
        rows.append(string_blocks_clear(pad(s, cap)) + ([] if clear is not None or pat is None else string_blocks_clear(pad(pat, args[1]))) + ext)
    out = simulate_rows(ir, rows)
    for (s, pat, want, ext), o in zip(cases, out):
        count, parts = split_out(o, nd, cap, P)
        assert count == len(want), (op, args, clear, s, pat, ext, count, want)
        assert parts == [pad(w, cap) for w in want] + [pad(b"", cap)] * (P - len(want)), (op, args, clear, s, pat, ext, parts, want)


CAP = 6
HAYS = [b"", b"a", b"aaaaaa", b"babab", b"ababab", b"a,b,,c", b"A..B..", b"ab ab", b"xyz"]
PADDED = [b"", b"a", b"aa", b"ab", b"aba", b"bab", b",", b"."]          # each at every capacity from its length to 3
CLEAR = ["a", "aa", "ab", "aba", "bab", ",", "."]                        # self-overlapping "aa", "aba", "bab"


def pattern_specs():
    for p in PADDED:
        for cp in range(len(p), 4):
            yield f"padded{cp}-{p.decode() or 'empty'}", p, cp, None
    for c in CLEAR:
        yield f"clear-{c}", c.encode(), len(c), c


SPECS = list(pattern_specs())
IDS = [s[0] for s in SPECS]
REFS = {"pstring_rsplit": rs_rsplitn, "pstring_split_terminator": rs_split_terminator, "pstring_rsplit_terminator": rs_rsplit_terminator,
        "pstring_split_inclusive": rs_split_inclusive}


@pytest.mark.parametrize("spec", SPECS, ids=IDS)
def test_split_family_clear_simulation(spec):
    _, pat, cp, clear = spec
    M = max_matches(CAP, len(pat) if clear else 0)
    for op, ref in REFS.items():
        check_split_rows(op, (CAP, cp), clear, CAP, M + 1, [(s, pat, ref(s, pat), []) for s in HAYS])
    for n in range(M + 3):
        check_split_rows("pstring_rsplitn", (CAP, cp, n), clear, CAP, min(M + 1, n), [(s, pat, rs_rsplitn(s, pat, n), []) for s in HAYS])


@pytest.mark.parametrize("spec", SPECS, ids=IDS)
def test_secret_count_clear_simulation(spec):
    """splitn_enc / rsplitn_enc / replacen_enc with n / count 0 ..= M + 2 and 65535, at count_blocks 1, 2 and 8"""
    _, pat, cp, clear = spec
    M = max_matches(CAP, len(pat) if clear else 0)
    to, cap_to = b"<>", 2
    for nb in (1, 2, 8):
        counts = [v for v in list(range(M + 3)) + [65535] if v < 4 ** nb]
        for op, ref in (("pstring_splitn_enc", rs_splitn), ("pstring_rsplitn_enc", rs_rsplitn)):
            check_split_rows(op, (CAP, cp, nb), clear, CAP, M + 1, [(s, pat, ref(s, pat, v), radix(v, nb)) for s in HAYS for v in counts])
        prog, ir = build("pstring_replacen_enc", (CAP, cp, cap_to, nb), clear)
        C = CAP + M * max(0, cap_to - (len(pat) if clear else 0))
        assert prog.n_outputs == 4 * C
        rows, want = [], []
        for s in HAYS:
            for v in counts:
                rows.append(string_blocks_clear(pad(s, CAP)) + ([] if clear else string_blocks_clear(pad(pat, cp))) +
                            string_blocks_clear(pad(to, cap_to)) + radix(v, nb))
                want.append(pad(rs_replacen(s, pat, to, v), C))
        for o, w in zip(simulate_rows(ir, rows), want):
            got = to_bytes(o)
            assert got == w and well_formed(got), ("pstring_replacen_enc", pat, cp, nb, got, w)


def test_split_ascii_whitespace_clear_simulation():
    hays = [b"", b" ", b"a", b"a b c", b" ab  c", b"\t\n\x0c\r x", b"a\x0bb c", b"abcdef", b"  \x0b  ", b"x y z"]
    for cap in (0, 1, 5, 6):
        cases = [(s, None, rs_split_ascii_whitespace(s), []) for s in hays if len(s) <= cap]
        check_split_rows("pstring_split_ascii_whitespace", (cap,), None, cap, (cap + 1) // 2, cases)


def test_repeat_enc_clear_simulation():
    for cap, max_count in ((3, 4), (2, 1), (0, 3), (3, 0)):
        for nb in (1, 2, 8):
            prog, ir = build("pstring_repeat_enc", (cap, max_count, nb))
            assert prog.n_outputs == 4 * cap * max_count
            counts = [v for v in list(range(max_count + 3)) + [65535] if v < 4 ** nb]
            strs = [s for s in (b"", b"a", b"xyz", b"ab") if len(s) <= cap]
            rows = [string_blocks_clear(pad(s, cap)) + radix(v, nb) for s in strs for v in counts]
            want = [pad(s * min(v, max_count), cap * max_count) for s in strs for v in counts]
            for o, w in zip(simulate_rows(ir, rows), want):
                assert to_bytes(o) == w, (cap, max_count, nb, to_bytes(o), w)


def test_strip_with_padded_pattern_clear_simulation():
    hays = [b"", b"a", b"ab", b"abab", b"aab", b"ba", b"abcabc"]
    for cp in (0, 1, 2, 3):
        pats = [p for p in (b"", b"a", b"ab", b"b", b"abc", b"ba") if len(p) <= cp]
        for op in ("pstring_strip_prefix", "pstring_strip_suffix"):
            prog, ir = build(op, (CAP, cp))
            assert prog.n_outputs == 1 + 4 * CAP
            cases = [(s, p) for s in hays for p in pats]
            out = simulate_rows(ir, [string_blocks_clear(pad(s, CAP)) + string_blocks_clear(pad(p, cp)) for s, p in cases])
            for (s, p), o in zip(cases, out):
                hit = s.startswith(p) if op == "pstring_strip_prefix" else s.endswith(p)
                rest = (s[len(p):] if op == "pstring_strip_prefix" else s[:len(s) - len(p)]) if hit else s
                assert (int(o[0]), to_bytes(o[1:])) == (int(hit), pad(rest, CAP)), (op, cp, s, p)


def test_eq_ignore_case_clear_simulation():
    words = [b"", b"a", b"A", b"Ab", b"aB", b"ab@", b"AB[", b"zZz", b"[`{", b"@"]
    for ca, cb in ((4, 4), (4, 2), (3, 5), (0, 2)):
        prog, ir = build("pstring_eq_ignore_case", (ca, cb))
        cases = [(a, b) for a in words for b in words if len(a) <= ca and len(b) <= cb]
        out = simulate_rows(ir, [string_blocks_clear(pad(a, ca)) + string_blocks_clear(pad(b, cb)) for a, b in cases])
        for (a, b), o in zip(cases, out):
            assert int(o[0]) == int(a.lower() == b.lower()), (ca, cb, a, b)
    prog, ir = build("pstring_eq_ignore_case", (4, 3), "AbC")
    out = simulate_rows(ir, [string_blocks_clear(pad(a, 4)) for a in words if len(a) <= 4])
    assert [int(o[0]) for o in out] == [int(a.lower() == b"abc") for a in words if len(a) <= 4]


def test_shapes():
    # the documented output counts, empty capacities included
    assert Program("pstring_rsplit", (0, 0)).n_outputs == digits_for(2)
    assert Program("pstring_split_inclusive", (4, 2), clear="ab").n_outputs == digits_for(3) + 4 * 4 * 3
    assert Program("pstring_rsplitn", (6, 2, 0)).n_outputs == 1
    assert Program("pstring_rsplit_terminator", (4, 5), clear="abcde").n_outputs == 1 + 16      # no match fits: one part
    assert Program("pstring_split_ascii_whitespace", (0,)).n_outputs == 1
    assert Program("pstring_split_ascii_whitespace", (7,)).n_outputs == digits_for(4) + 4 * 7 * 4
    assert Program("pstring_splitn_enc", (6, 2, 3)).n_outputs == digits_for(8) + 4 * 6 * 8
    assert Program("pstring_repeat_enc", (3, 0, 2)).n_outputs == 0
    assert Program("pstring_replacen_enc", (6, 1, 3, 2)).n_outputs == 4 * (6 + 7 * 3)
    assert Program("pstring_strip_suffix", (6, 2)).n_outputs == 1 + 24 and Program("pstring_eq_ignore_case", (3, 5)).n_outputs == 1
    # the inputs: strings, then the secret integer
    assert Program("pstring_replacen_enc", (6, 2, 3, 5)).n_inputs == 4 * (6 + 2 + 3) + 5
    assert Program("pstring_rsplitn_enc", (6, 2, 4), clear="ab").n_inputs == 4 * 6 + 4
    # a clear pattern without a proper border needs no chain over positions
    assert Program("pstring_rsplit", (64, 2), clear="ab").n_levels < 64
    # larger programs keep the noise bound
    for op, args, clear in (("pstring_rsplit", (12, 4), None), ("pstring_rsplit_terminator", (12, 3), "aba"),
                            ("pstring_split_inclusive", (12, 4), None), ("pstring_splitn_enc", (12, 3, 8), None),
                            ("pstring_replacen_enc", (12, 4, 4, 3), None), ("pstring_split_ascii_whitespace", (16,), None),
                            ("pstring_repeat_enc", (4, 3, 8), None), ("pstring_strip_suffix", (12, 4), None)):
        build(op, args, clear)


NEW_OPS = [("pstring_rsplit", (6, 2)), ("pstring_rsplitn", (6, 2, 3)), ("pstring_split_terminator", (6, 2)),
           ("pstring_rsplit_terminator", (6, 2)), ("pstring_split_inclusive", (6, 2)), ("pstring_split_ascii_whitespace", (6,)),
           ("pstring_repeat_enc", (3, 2, 2)), ("pstring_replacen_enc", (6, 2, 2, 2)), ("pstring_splitn_enc", (6, 2, 2)),
           ("pstring_rsplitn_enc", (6, 2, 2)), ("pstring_strip_prefix", (6, 2)), ("pstring_strip_suffix", (6, 2)),
           ("pstring_eq_ignore_case", (4, 3))]


def test_argument_errors():
    for op, args in NEW_OPS:
        with pytest.raises(NativeError, match="expected"):
            Program(op, args[:-1] if op not in ("pstring_strip_prefix", "pstring_strip_suffix") else ())
    with pytest.raises(NativeError, match="clear pattern"):      # the one-argument strip without a clear pattern
        Program("pstring_strip_suffix", (8,))
    for op, args in (("pstring_repeat_enc", (3, 2, 0)), ("pstring_repeat_enc", (3, 2, 17)), ("pstring_replacen_enc", (6, 2, 2, 0)),
                     ("pstring_splitn_enc", (6, 2, 17)), ("pstring_rsplitn_enc", (6, 2, 0))):
        with pytest.raises(NativeError, match="1 ..= 16"):
            Program(op, args)
    for op, args in (("pstring_rsplit", (8, 3)), ("pstring_split_inclusive", (8, 1)), ("pstring_replacen_enc", (8, 0, 2, 2)),
                     ("pstring_eq_ignore_case", (4, 3))):
        with pytest.raises(NativeError, match="differs from the clear pattern's length"):
            Program(op, args, clear="ab")
    for op, args in (("pstring_split_ascii_whitespace", (6,)), ("pstring_repeat_enc", (3, 2, 2))):
        with pytest.raises(NativeError, match="no clear operand"):
            Program(op, args, clear="ab")
    for op, args in (("pstring_rsplit", (2**40, 1)), ("pstring_strip_prefix", (8, 2**21)), ("pstring_repeat_enc", (4, 2**60, 2)),
                     ("pstring_eq_ignore_case", (2**21, 1))):
        with pytest.raises(NativeError, match="limited"):
            Program(op, args)
    for op, args in (("pstring_rsplit", (2**10, 1)), ("pstring_split_ascii_whitespace", (2**11,)), ("pstring_repeat_enc", (2**10, 2**11, 2)),
                     ("pstring_replacen_enc", (2**19, 0, 2**19, 2)), ("pstring_rsplitn", (2**10, 0, 2**10 + 1))):
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


def test_split_family_with_real_pbs_toy(orc, toy_keys):
    """small programs executed with the oracle's CPU KS-PBS on the toy parameter set"""
    from oracle import radix as R
    p, ck, sk = toy_keys
    prm = engine_params(p)
    enc = lambda *xs: np.concatenate([R.encrypt_string(ck, pad(x, c)) for x, c in xs])
    enc_int = lambda v, nb: np.stack(R.encrypt_radix(ck, v, nb))
    cap = 4
    out = R.run_program(Program("pstring_rsplit", (cap, 2), params=prm).ir(), sk, enc((b"a,bc", cap), (b",", 2)))
    nd = digits_for(cap + 2)
    assert R.decrypt_radix(ck, out[:nd]) == 2
    assert [R.decrypt_string(ck, out[nd + 16 * k: nd + 16 * (k + 1)]) for k in range(cap + 2)] == [pad(b"bc", 4), pad(b"a", 4)] + [pad(b"", 4)] * 4
    out = R.run_program(Program("pstring_split_inclusive", (cap, 1), clear=",", params=prm).ir(), sk, enc((b"a,b,", cap)))
    nd = digits_for(cap + 1)
    assert R.decrypt_radix(ck, out[:nd]) == 2
    assert [R.decrypt_string(ck, out[nd + 16 * k: nd + 16 * (k + 1)]) for k in range(2)] == [pad(b"a,", 4), pad(b"b,", 4)]
    out = R.run_program(Program("pstring_splitn_enc", (3, 1, 2), params=prm).ir(), sk, np.concatenate([enc((b"a-b", 3), (b"-", 1)), enc_int(1, 2)]))
    nd = digits_for(5)
    assert R.decrypt_radix(ck, out[:nd]) == 1 and R.decrypt_string(ck, out[nd:nd + 12]) == pad(b"a-b", 3)
