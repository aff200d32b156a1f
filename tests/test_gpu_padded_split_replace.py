"""GPU test (-m gpu) of the null-padded replace / replacen / split / splitn / split_once / rsplit_once at PARAM_MESSAGE_2_CARRY_2_KS_PBS
with real keys: decrypted results against Rust's str semantics (host/padded.h), and the cost of replace / split at capacity 32."""
import numpy as np
import pytest

from fhe_string_bounty_b200.host import Program
from helpers import engine_params
from test_padded_split_replace import digits_for, max_matches, pad, rs_replacen, rs_split_once, rs_splitn

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu(orc, keys_2_2):
    import fhe_string_bounty_b200 as F
    p, ck, sk = keys_2_2
    eng = F.Engine(engine_params(p))
    eng.upload_ksk(sk.ksk)
    eng.upload_bsk_std(sk.bsk)
    yield eng, ck, engine_params(p)
    eng.close()


def enc(ck, *strings):
    from oracle import radix as R
    return np.concatenate([R.encrypt_string(ck, pad(s, c)) for s, c in strings])


CAP = 12


def test_replace_gpu(gpu):
    from oracle import radix as R
    eng, ck, prm = gpu
    P = Program("pstring_replace", (CAP, 3, 3), params=prm)                    # padded `from`
    for s, frm, to in ((b"aaaaa", b"aa", b"<>"), (b"ab cd ab", b"", b"."), (b"encrypted", b"pt", b"PT!"), (b"xyz", b"q", b"")):
        C = CAP + max_matches(CAP, 0) * 3
        assert R.decrypt_string(ck, P.run(eng, enc(ck, (s, CAP), (frm, 3), (to, 3)))) == pad(rs_replacen(s, frm, to), C), (s, frm, to)
    P = Program("pstring_replacen", (CAP, 3, 2, 2), clear="aba", params=prm)    # clear `from` that overlaps itself
    for s in (b"abababababa", b"aba", b"xx"):                                  # `to` is shorter than the pattern: C == CAP
        assert R.decrypt_string(ck, P.run(eng, enc(ck, (s, CAP), (b"Z", 2)))) == pad(rs_replacen(s, b"aba", b"Z", 2), CAP), s


def test_split_gpu(gpu):
    from oracle import radix as R
    eng, ck, prm = gpu
    dec = ck.decrypt_message_and_carry
    for op, args, clear, n in (("pstring_split", (CAP, 2), None, None), ("pstring_splitn", (CAP, 2, 3), None, 3),
                               ("pstring_split", (CAP, 2), ", ", None)):
        P = Program(op, args, clear=clear, params=prm)
        Pn = min(max_matches(CAP, len(clear) if clear else 0) + 1, n or 10**9)
        nd = digits_for(Pn)
        for s, pat in ((b"a, b,, c", b", "), (b"aaaaa", b"aa"), (b"abc", b"")):
            if clear and pat != clear.encode():
                continue
            out = P.run(eng, enc(ck, (s, CAP)) if clear else enc(ck, (s, CAP), (pat, 2)))
            want = rs_splitn(s, pat, n)
            assert R.decrypt_radix(ck, out[:nd]) == len(want), (op, s, pat)
            parts = [R.decrypt_string(ck, out[nd + 4 * CAP * k: nd + 4 * CAP * (k + 1)]) for k in range(Pn)]
            assert parts == [pad(w, CAP) for w in want] + [pad(b"", CAP)] * (Pn - len(want)), (op, s, pat)
    for op, last in (("pstring_split_once", False), ("pstring_rsplit_once", True)):
        P = Program(op, (CAP, 3), params=prm)
        for s, pat in ((b"key=val=x", b"="), (b"aaaa", b"aa"), (b"abc", b""), (b"abc", b"zz")):
            out = P.run(eng, enc(ck, (s, CAP), (pat, 3)))
            want = rs_split_once(s, pat, last)
            got = (dec(out[0]), R.decrypt_string(ck, out[1:1 + 4 * CAP]), R.decrypt_string(ck, out[1 + 4 * CAP:]))
            assert got == ((1, pad(want[0], CAP), pad(want[1], CAP)) if want else (0, pad(b"", CAP), pad(b"", CAP))), (op, s, pat, got)


def test_split_replace_cost_gpu(gpu):
    """PBS count, levels and device time of replace / split at capacity 32, with a clear "ab" and a padded pattern of capacity 4"""
    from oracle import radix as R
    eng, ck, prm = gpu
    s = b"ab cd ab ef abab gh ab ijk ab xy"
    for op, args, clear in (("pstring_replace", (32, 2, 2), "ab"), ("pstring_replace", (32, 4, 4), None),
                            ("pstring_split", (32, 2), "ab"), ("pstring_split", (32, 4), None)):
        P = Program(op, args, clear=clear, params=prm)
        ins = [(s, 32)] + ([] if clear else [(b"ab", 4)]) + ([(b"XY", args[2])] if op == "pstring_replace" else [])
        x = enc(ck, *ins)
        out = P.run(eng, x)
        ms = []
        for _ in range(3):
            P.run(eng, x)
            ms.append(P.last_ms())
        if op == "pstring_replace":
            C = 32 + max_matches(32, len(clear) if clear else 0) * (args[2] - (len(clear) if clear else 0))
            assert R.decrypt_string(ck, out) == pad(s.replace(b"ab", b"XY"), C)
        else:
            assert R.decrypt_radix(ck, out[:digits_for(max_matches(32, 2 if clear else 0) + 1)]) == len(s.split(b"ab"))
        print(f"{op} capacity 32, {'clear ' + repr(clear) if clear else 'padded pattern, capacity 4'}: {P.n_pbs} PBS in "
              f"{P.n_levels} levels, device {min(ms):.1f} ms (best of 3; {', '.join(f'{m:.1f}' for m in ms)})")
