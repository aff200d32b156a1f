"""Null-padded replace / replacen / split / splitn / split_once / rsplit_once (host/padded.h) on CPU.

The recorded programs are executed noise-free on plaintexts (simulate_program_clear) against a small reference of Rust's str semantics
(leftmost non-overlapping matches; the empty pattern matches at every char boundary 0 ..= len), with padded and clear patterns.  The
noise and depth bounds are read from the program IR, and a few small cases run through the CPU oracle's real KS-PBS on the toy keys."""
import numpy as np
import pytest

from fhe_string_bounty_b200 import NativeError
from fhe_string_bounty_b200.host import Program
from helpers import engine_params, simulate_program_clear, string_blocks_clear


# ---- reference: Rust's str methods with a &str pattern ------------------------------------------------------------------------------
def rs_matches(s: bytes, pat: bytes):
    """start indices of the leftmost non-overlapping matches (str::match_indices)"""
    if not pat:
        return list(range(len(s) + 1))
    out, i = [], 0
    while (j := s.find(pat, i)) >= 0:
        out.append(j)
        i = j + len(pat)
    return out


def rs_replacen(s, pat, to, count=None):
    ms = rs_matches(s, pat)[:count]
    out, last = b"", 0
    for m in ms:
        out += s[last:m] + to
        last = m + len(pat)
    return out + s[last:]


def rs_splitn(s, pat, n=None):
    if n == 0:
        return []
    ms = rs_matches(s, pat)
    if n is not None:
        ms = ms[:n - 1]
    parts, last = [], 0
    for m in ms:
        parts.append(s[last:m])
        last = m + len(pat)
    return parts + [s[last:]]


def rs_split_once(s, pat, last=False):
    ms = rs_matches(s, pat)
    if not pat and last:
        ms = [len(s)]                                 # rfind("") == len
    elif last and ms:
        ms = [s.rfind(pat)]                           # rsplit_once splits at rfind, which may overlap an earlier match
    if not ms:
        return None
    return s[:ms[0]], s[ms[0] + len(pat):]


def test_reference_against_python():
    words = [b"", b"a", b"aa", b"aaa", b"aaaaa", b"ababa", b"abcab", b"a,b,,c", b"xyz", b", x, "]
    pats = [b"a", b"aa", b"ab", b"aba", b",", b", ", b"x", b"zz"]
    for s in words:
        for p in pats:
            assert rs_replacen(s, p, b"<>") == s.replace(p, b"<>")
            for c in range(4):
                assert rs_replacen(s, p, b"-", c) == s.replace(p, b"-", c)
            assert rs_splitn(s, p) == s.split(p)
            for n in range(1, 4):
                assert rs_splitn(s, p, n) == s.split(p, n - 1)
            a, sep, b = s.partition(p)
            assert rs_split_once(s, p) == ((a, b) if sep else None)
            a, sep, b = s.rpartition(p)
            assert rs_split_once(s, p, last=True) == ((a, b) if sep else None)
    # the empty pattern, as Rust has it
    assert rs_replacen(b"ab", b"", b"x") == b"xaxbx"
    assert rs_replacen(b"ab", b"", b"x", 2) == b"xaxb"
    assert rs_splitn(b"ab", b"") == [b"", b"a", b"b", b""]
    assert rs_splitn(b"ab", b"", 2) == [b"", b"ab"]
    assert rs_splitn(b"", b"") == [b"", b""]
    assert rs_split_once(b"ab", b"") == (b"", b"ab") and rs_split_once(b"ab", b"", last=True) == (b"ab", b"")
    # non-overlapping, left to right
    assert rs_replacen(b"aaaa", b"aa", b"b") == b"bb" and rs_splitn(b"aaa", b"aa") == [b"", b"a"]
    assert rs_split_once(b"aaa", b"aa", last=True) == (b"a", b"")


# ---- the recorded programs ------------------------------------------------------------------------------------------------------------
def pad(s: bytes, cap: int) -> bytes:
    assert len(s) <= cap
    return s + b"\0" * (cap - len(s))


def to_bytes(blocks) -> bytes:
    return bytes(sum(int(d) << (2 * i) for i, d in enumerate(blocks[k:k + 4])) for k in range(0, len(blocks), 4))


def to_int(blocks) -> int:
    return sum(int(d) << (2 * i) for i, d in enumerate(blocks))


def digits_for(v):
    d = 1
    while 4 ** d <= v:
        d += 1
    return d


def max_matches(cap, m_min):
    return cap + 1 if m_min == 0 else cap // m_min


def well_formed(b: bytes) -> bool:
    """zero bytes only after the content"""
    return b"\0" not in b.rstrip(b"\0")


def run(op, args, ins, clear=None):
    P = Program(op, args, clear=clear)
    ir = P.ir()
    out, hits = simulate_program_clear(ir, ins, 16)
    assert hits == 0, (op, args, hits)
    # every result block is a PBS output or trivial: it can feed any other operation
    assert int(ir.output_degree_noise[:, 1].max(initial=0)) <= 1 and int(ir.output_degree_noise[:, 0].max(initial=0)) <= 3
    return out, P


def pbs_input_noise(ir) -> int:
    """largest nominal noise of a PBS input: inputs and PBS outputs are 1, a leveled instruction is sum |coef| * noise"""
    noise = np.zeros(ir.n_slots, dtype=np.int64)
    noise[: ir.n_inputs] = 1
    worst = 0
    for lv in range(len(ir.level_lin_off) - 1):
        for li in range(int(ir.level_lin_off[lv]), int(ir.level_lin_off[lv + 1])):
            out, tb, te = (int(v) for v in ir.lin[li])
            noise[out] = int(np.sum(np.abs(ir.term_coef[tb:te]) * noise[ir.term_slot[tb:te]]))
        p0, p1 = int(ir.level_pbs_off[lv]), int(ir.level_pbs_off[lv + 1])
        if p1 > p0:
            worst = max(worst, int(noise[ir.pbs[p0:p1, 0]].max()))
            noise[ir.pbs[p0:p1, 1]] = 1
    return worst


def inputs(s, cap, pat=None, cap_pat=None, to=None, cap_to=None):
    ins = string_blocks_clear(pad(s, cap))
    if pat is not None:
        ins += string_blocks_clear(pad(pat, cap_pat))
    if to is not None:
        ins += string_blocks_clear(pad(to, cap_to))
    return ins


def check_replace(s, cap, frm, cap_from, to, cap_to, count=None, clear=False):
    m_min = len(frm) if clear else 0
    M = max_matches(cap, m_min)
    n_rep = M if count is None else min(count, M)
    C = cap + n_rep * max(0, cap_to - m_min)
    op, args = ("pstring_replace", (cap, cap_from, cap_to)) if count is None else ("pstring_replacen", (cap, cap_from, cap_to, count))
    ins = inputs(s, cap, None if clear else frm, cap_from, to, cap_to)
    out, P = run(op, args, ins, clear=frm if clear else None)
    assert P.n_outputs == 4 * C
    got = to_bytes(out)
    assert got == pad(rs_replacen(s, frm, to, count), C), (op, s, frm, to, count, clear, got)
    assert well_formed(got)


def check_split(s, cap, pat, cap_pat, n=None, clear=False):
    M = max_matches(cap, len(pat) if clear else 0)
    Pn = M + 1 if n is None else min(M + 1, n)
    nd = digits_for(Pn)
    op, args = ("pstring_split", (cap, cap_pat)) if n is None else ("pstring_splitn", (cap, cap_pat, n))
    out, P = run(op, args, inputs(s, cap, None if clear else pat, cap_pat), clear=pat if clear else None)
    assert P.n_outputs == nd + 4 * cap * Pn
    want = rs_splitn(s, pat, n)
    assert to_int(out[:nd]) == len(want), (op, s, pat, n, clear)
    parts = [to_bytes(out[nd + 4 * cap * k: nd + 4 * cap * (k + 1)]) for k in range(Pn)]
    assert parts == [pad(w, cap) for w in want] + [pad(b"", cap)] * (Pn - len(want)), (op, s, pat, n, clear, parts)


def check_split_once(s, cap, pat, cap_pat, clear=False):
    for op, last in (("pstring_split_once", False), ("pstring_rsplit_once", True)):
        out, P = run(op, (cap, cap_pat), inputs(s, cap, None if clear else pat, cap_pat), clear=pat if clear else None)
        assert P.n_outputs == 1 + 8 * cap
        want = rs_split_once(s, pat, last)
        got = (int(out[0]), to_bytes(out[1:1 + 4 * cap]), to_bytes(out[1 + 4 * cap:]))
        assert got == ((1, pad(want[0], cap), pad(want[1], cap)) if want else (0, pad(b"", cap), pad(b"", cap))), (op, s, pat, clear, got)


CAP = 7
HAYS = [b"", b"aaaaa", b"ababa", b"abcabca", b"xabx", b"a,b,,c", b"zzzzzzz"]     # empty; matches at the start, at the end, back to back;
PATS = [b"", b"a", b"aa", b"ab", b"aba", b"ca", b"abcabcab"]                    # a haystack that fills its capacity; overlapping patterns;
TOS = [b"", b"-", b"<<<"]                                                       # a pattern longer than the haystack; the empty pattern


@pytest.mark.parametrize("clear", [False, True], ids=["padded", "clear"])
@pytest.mark.parametrize("frm", PATS)
def test_replace_clear_simulation(frm, clear):
    cap_from = len(frm) if clear else 3
    if len(frm) > cap_from:
        cap_from = len(frm)
    for s in HAYS:
        for to in TOS:                                                          # empty, longer than `from`, filling its capacity
            check_replace(s, CAP, frm, cap_from, to, 3, clear=clear)
        for count in (0, 1, 2, 9):
            check_replace(s, CAP, frm, cap_from, b"<<<", 3, count=count, clear=clear)


@pytest.mark.parametrize("clear", [False, True], ids=["padded", "clear"])
@pytest.mark.parametrize("pat", PATS)
def test_split_clear_simulation(pat, clear):
    cap_pat = len(pat) if clear else max(3, len(pat))
    for s in HAYS:
        check_split(s, CAP, pat, cap_pat, clear=clear)
        for n in (0, 1, 2, 9):
            check_split(s, CAP, pat, cap_pat, n=n, clear=clear)
        check_split_once(s, CAP, pat, cap_pat, clear=clear)


def test_shapes_noise_and_depth():
    # a clear pattern without a proper border needs no chain over positions: well under one level per position
    for op, args in (("pstring_replace", (128, 2, 2)), ("pstring_split", (128, 2))):
        P = Program(op, args, clear="ab")
        assert P.n_levels < 128, (op, P.n_levels)
    # no PBS input above the 15 nominal noise units of a count tree
    cases = [("pstring_replace", (12, 4, 4), None), ("pstring_replace", (12, 2, 3), "aa"), ("pstring_replacen", (12, 4, 4, 2), None),
             ("pstring_replacen", (12, 3, 2, 1), "aba"), ("pstring_split", (12, 4), None), ("pstring_split", (12, 2), ", "),
             ("pstring_splitn", (12, 4, 3), None), ("pstring_split_once", (12, 4), None), ("pstring_rsplit_once", (12, 2), "ab"),
             ("pstring_split", (20, 18), None), ("pstring_replace", (20, 17, 2), None)]
    for op, args, clear in cases:
        assert pbs_input_noise(Program(op, args, clear=clear).ir()) <= 15, (op, args, clear)
    # the documented output counts hold for empty capacities too
    assert Program("pstring_replace", (0, 0, 2)).n_outputs == 4 * 2          # "".replace("", to) == to
    assert Program("pstring_split", (0, 0)).n_outputs == digits_for(2)
    assert Program("pstring_splitn", (6, 2, 0)).n_outputs == 1
    assert Program("pstring_replace", (4, 5, 3), clear="abcde").n_outputs == 16    # a pattern longer than the haystack: no match fits


def test_argument_errors():
    for op, args in (("pstring_replace", (8, 2)), ("pstring_replacen", (8, 2, 2)), ("pstring_split", (8,)), ("pstring_splitn", (8, 2)),
                     ("pstring_split_once", (8,)), ("pstring_rsplit_once", ())):
        with pytest.raises(NativeError, match="expected"):
            Program(op, args)
    with pytest.raises(NativeError, match="differs from the clear pattern's length"):
        Program("pstring_split", (8, 3), clear="ab")
    with pytest.raises(NativeError, match="differs from the clear pattern's length"):
        Program("pstring_replace", (8, 0, 2), clear="a")
    with pytest.raises(NativeError, match="exceed"):
        Program("pstring_replace", (2**19, 0, 2**19))
    with pytest.raises(NativeError, match="limited"):
        Program("pstring_split", (2**40, 1))


def test_split_replace_with_real_pbs_toy(orc, toy_keys):
    """small programs executed with the oracle's CPU KS-PBS on the toy parameter set"""
    from oracle import radix as R
    p, ck, sk = toy_keys
    prm = engine_params(p)
    cap = 4
    enc = lambda *xs: np.concatenate([R.encrypt_string(ck, pad(x, c)) for x, c in xs])
    out = R.run_program(Program("pstring_replace", (cap, 2, 2), clear="ab", params=prm).ir(), sk, enc((b"abab", cap), (b"x", 2)))
    assert R.decrypt_string(ck, out) == pad(b"xx", 4)
    out = R.run_program(Program("pstring_split", (cap, 1), params=prm).ir(), sk, enc((b"a,b", cap), (b",", 1)))
    nd = digits_for(cap + 2)
    assert R.decrypt_radix(ck, out[:nd]) == 2
    assert [R.decrypt_string(ck, out[nd + 4 * cap * k: nd + 4 * cap * (k + 1)]) for k in range(3)] == [pad(b"a", 4), pad(b"b", 4), pad(b"", 4)]
    out = R.run_program(Program("pstring_rsplit_once", (3, 2), params=prm).ir(), sk, enc((b"aaa", 3), (b"aa", 2)))
    assert ck.decrypt_message_and_carry(out[0]) == 1
    assert (R.decrypt_string(ck, out[1:13]), R.decrypt_string(ck, out[13:])) == (pad(b"a", 3), pad(b"", 3))
