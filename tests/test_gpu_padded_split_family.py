"""GPU test (-m gpu) of the null-padded rsplit / rsplitn / split_terminator / rsplit_terminator / split_inclusive / split_ascii_whitespace,
the secret-count ops (repeat_enc, replacen_enc, splitn_enc, rsplitn_enc), strip_prefix / strip_suffix with a padded pattern and the padded
eq_ignore_case at PARAM_MESSAGE_2_CARRY_2_KS_PBS: decrypted results with real keys against Rust's str semantics (host/padded.h), three of
them word for word against the exact executor on the coarse lattice, rsplit on two ranks of one GPU, and the cost at capacity 32."""
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from fhe_string_bounty_b200.host import Program
from helpers import coarse_inputs, engine_params, round_to_lattice
from test_gpu_exact_programs import ExactPrograms, _run_device, coarse_keys
from test_padded_split_family import (rs_rsplit_terminator, rs_rsplitn, rs_split_ascii_whitespace, rs_split_inclusive,
                                      rs_split_terminator)
from test_padded_split_replace import digits_for, max_matches, pad, rs_replacen, rs_splitn

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


def enc_int(ck, v, nb):
    from oracle import radix as R
    return np.stack(R.encrypt_radix(ck, v, nb))


def decrypt_split(ck, out, nd, cap, P):
    from oracle import radix as R
    return R.decrypt_radix(ck, out[:nd]), [R.decrypt_string(ck, out[nd + 4 * cap * k: nd + 4 * cap * (k + 1)]) for k in range(P)]


def assert_split(ck, out, cap, P, want, label):
    count, parts = decrypt_split(ck, out, digits_for(P), cap, P)
    assert count == len(want), (label, count, want)
    assert parts == [pad(w, cap) for w in want] + [pad(b"", cap)] * (P - len(want)), (label, parts, want)


CAP = 12
HAYS = [(b"A..B..", b"."), (b"babababab", b"bab"), (b"a,b,,c,", b","), (b"ab", b""), (b"", b"x"), (b"no match", b"zz")]


def test_split_family_gpu(gpu):
    eng, ck, prm = gpu
    M = max_matches(CAP, 0)
    for op, ref in (("pstring_rsplit", rs_rsplitn), ("pstring_split_terminator", rs_split_terminator),
                    ("pstring_rsplit_terminator", rs_rsplit_terminator), ("pstring_split_inclusive", rs_split_inclusive)):
        P = Program(op, (CAP, 3), params=prm)                                    # padded pattern
        for s, pat in HAYS:
            assert_split(ck, P.run(eng, enc(ck, (s, CAP), (pat, 3))), CAP, M + 1, ref(s, pat), (op, s, pat))
    P = Program("pstring_rsplitn", (CAP, 3, 3), params=prm)
    for s, pat in HAYS:
        assert_split(ck, P.run(eng, enc(ck, (s, CAP), (pat, 3))), CAP, 3, rs_rsplitn(s, pat, 3), ("rsplitn", s, pat))
    Mc = max_matches(CAP, 3)
    P = Program("pstring_rsplit", (CAP, 3), clear="bab", params=prm)            # a clear pattern that overlaps itself
    for s in (b"babababab", b"bab", b"xbabbab"):
        assert_split(ck, P.run(eng, enc(ck, (s, CAP))), CAP, Mc + 1, rs_rsplitn(s, b"bab"), ("rsplit clear", s))
    P = Program("pstring_split_ascii_whitespace", (CAP,), params=prm)
    for s in (b" a\tbc \x0bd\n", b"", b"one two thre", b"   "):
        assert_split(ck, P.run(eng, enc(ck, (s, CAP))), CAP, (CAP + 1) // 2, rs_split_ascii_whitespace(s), ("split_ascii_whitespace", s))


def test_secret_counts_gpu(gpu):
    """encrypted counts 0, 1, M, M + 1 and 65535 (8 blocks)"""
    from oracle import radix as R
    eng, ck, prm = gpu
    M = max_matches(CAP, 0)
    s, pat = b"a,b,,c,d", b","
    for op, ref in (("pstring_splitn_enc", rs_splitn), ("pstring_rsplitn_enc", rs_rsplitn)):
        P = Program(op, (CAP, 2, 8), params=prm)
        for v in (0, 1, 3, M, M + 1, 65535):
            x = np.concatenate([enc(ck, (s, CAP), (pat, 2)), enc_int(ck, v, 8)])
            assert_split(ck, P.run(eng, x), CAP, M + 1, ref(s, pat, v), (op, v))
    P = Program("pstring_replacen_enc", (CAP, 2, 2, 8), params=prm)
    C = CAP + M * 2
    for v in (0, 1, 2, M, M + 1, 65535):
        x = np.concatenate([enc(ck, (s, CAP), (pat, 2), (b"<>", 2)), enc_int(ck, v, 8)])
        assert R.decrypt_string(ck, P.run(eng, x)) == pad(rs_replacen(s, pat, b"<>", v), C), ("replacen_enc", v)
    P = Program("pstring_repeat_enc", (4, 3, 8), params=prm)
    for v in (0, 1, 3, 4, 65535):
        x = np.concatenate([enc(ck, (b"ab", 4)), enc_int(ck, v, 8)])
        assert R.decrypt_string(ck, P.run(eng, x)) == pad(b"ab" * min(v, 3), 12), ("repeat_enc", v)


def test_strip_and_eq_ignore_case_gpu(gpu):
    from oracle import radix as R
    eng, ck, prm = gpu
    dec = ck.decrypt_message_and_carry
    for op in ("pstring_strip_prefix", "pstring_strip_suffix"):
        P = Program(op, (CAP, 3), params=prm)
        for s, pat in ((b"prefix-rest", b"pre"), (b"a.tar.gz", b".gz"), (b"abc", b""), (b"abc", b"x"), (b"", b"ab")):
            hit = s.startswith(pat) if op == "pstring_strip_prefix" else s.endswith(pat)
            rest = (s[len(pat):] if op == "pstring_strip_prefix" else s[:len(s) - len(pat)]) if hit else s
            out = P.run(eng, enc(ck, (s, CAP), (pat, 3)))
            assert (dec(out[0]), R.decrypt_string(ck, out[1:])) == (int(hit), pad(rest, CAP)), (op, s, pat)
    P = Program("pstring_eq_ignore_case", (CAP, 8), params=prm)
    for a, b in ((b"Hello World", b"hELLO"), (b"Hello", b"hELLO"), (b"", b""), (b"a@", b"A`"), (b"Zz", b"zZ")):
        assert dec(P.run(eng, enc(ck, (a, CAP), (b, 8)))[0]) == int(a.lower() == b.lower()), (a, b)


# ---- word for word on the coarse lattice ----------------------------------------------------------------------------------------------
EXACT_SPECS = [("pstring_rsplit", (6, 2), None), ("pstring_split_inclusive", (6, 2), None), ("pstring_splitn_enc", (6, 2, 2), None)]


def test_exact_split_family(orc):
    progs = ExactPrograms(orc, "2_2", 0xF600, EXACT_SPECS)
    eng = progs.engine()
    progs.check(eng, "tuned, fused KS -> PBS", device=True)
    eng.close()


def test_rsplit_sharded_equals_run_device(orc):
    """pstring_rsplit {32, 4} on two ranks of one GPU (DeviceComm.local_group): every rank's words, rounded to the coarse lattice, equal
    program_run_device's"""
    import torch
    import fhe_string_bounty_b200 as F
    from fhe_string_bounty_b200 import multi_gpu as MG
    from helpers import coarse_shift
    p = orc.params("2_2")
    bsk, ksk = coarse_keys(orc, p, 0xF700)
    engines = []
    for _ in range(2):
        e = F.Engine(engine_params(p))
        e.upload_ksk(ksk)
        e.upload_bsk_std(bsk)
        engines.append(e)
    comms = MG.DeviceComm.local_group(engines)
    streams = [torch.cuda.Stream() for _ in comms]
    progs = [Program("pstring_rsplit", (32, 4), params=engine_params(p)) for _ in comms]
    x = coarse_inputs(p, progs[0].n_inputs, 0xF701)
    try:
        def one(r):
            with torch.cuda.stream(streams[r]):
                return comms[r].to_host(MG.run_program_sharded(comms[r], progs[r], x)).copy()
        with ThreadPoolExecutor(2) as pool:
            got = list(pool.map(one, range(2)))
        plan = progs[0].shard_plan(2, comms[0].min_shard_width)
        want = _run_device(engines[0], Program("pstring_rsplit", (32, 4), params=engine_params(p)), x)
    finally:
        for c in comms:
            c.close()
        for e in engines:
            e.close()
    u = coarse_shift(p)
    assert plan[0] > 0, "nothing split"
    assert np.array_equal(got[0], got[1])
    bad = round_to_lattice(got[0], u) != round_to_lattice(want, u)
    print(f"pstring_rsplit(32, 4) at world 2 on one GPU: {plan[0]} split levels, {got[0].size} output words, {int(bad.sum())} differ from "
          f"program_run_device on the 2^{u} lattice; raw words identical: {np.array_equal(got[0], want)}")
    assert not bad.any()


# ---- cost -------------------------------------------------------------------------------------------------------------------------------
def test_split_family_cost_gpu(gpu):
    """PBS count, levels and best-of-3 device time at capacity 32"""
    from oracle import radix as R
    eng, ck, prm = gpu
    s = b"ab cd ab ef abab gh ab ijk ab xy"
    cases = [("pstring_rsplit", (32, 2), "ab", [(s, 32)], lambda out: decrypt_split(ck, out, digits_for(17), 32, 17)[0] == len(s.split(b"ab"))),
             ("pstring_rsplit", (32, 4), None, [(s, 32), (b"ab", 4)],
              lambda out: decrypt_split(ck, out, digits_for(34), 32, 34)[0] == len(s.split(b"ab"))),
             ("pstring_split_inclusive", (32, 4), None, [(s, 32), (b"ab", 4)],
              lambda out: decrypt_split(ck, out, digits_for(34), 32, 34)[0] == len(rs_split_inclusive(s, b"ab"))),
             ("pstring_split_ascii_whitespace", (32,), None, [(s, 32)],
              lambda out: decrypt_split(ck, out, digits_for(16), 32, 16)[0] == len(s.split())),
             ("pstring_replacen_enc", (32, 4, 4, 8), None, [(s, 32), (b"ab", 4), (b"XY!", 4)],
              lambda out: R.decrypt_string(ck, out) == pad(s.replace(b"ab", b"XY!", 3), 32 + 33 * 4)),
             ("pstring_repeat_enc", (8, 4, 8), None, [(b"abc", 8)], lambda out: R.decrypt_string(ck, out) == pad(b"abc" * 3, 32))]
    for op, args, clear, strings, ok in cases:
        P = Program(op, args, clear=clear, params=prm)
        x = enc(ck, *strings)
        if op.endswith("_enc"):
            x = np.concatenate([x, enc_int(ck, 3, 8)])
        out = P.run(eng, x)
        assert ok(out), (op, args, clear)
        ms = []
        for _ in range(3):
            P.run(eng, x)
            ms.append(P.last_ms())
        print(f"{op}{args}{', clear ' + repr(clear) if clear else ''}: {P.n_pbs} PBS in {P.n_levels} levels, "
              f"device {min(ms):.1f} ms (best of 3; {', '.join(f'{m:.1f}' for m in ms)})")
