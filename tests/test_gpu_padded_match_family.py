"""GPU test (-m gpu) of the null-padded matches / match_indices / rmatch_indices / trim_start_matches / trim_end_matches / lines /
split_whitespace at PARAM_MESSAGE_2_CARRY_2_KS_PBS: decrypted results with real keys against Rust's str semantics (host/padded.h), three
of them word for word against the exact executor on the coarse lattice, rmatch_indices on two ranks of one GPU, and the cost at
capacity 32 with the card's name and power limit."""
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from fhe_string_bounty_b200.host import Program
from helpers import coarse_inputs, engine_params, round_to_lattice
from test_gpu_exact_programs import ExactPrograms, _run_device, coarse_keys
from test_gpu_padded_split_family import assert_split, enc
from test_padded_match_family import (rs_lines, rs_match_indices, rs_rmatch_indices, rs_split_whitespace, rs_trim_end_matches,
                                      rs_trim_start_matches)
from test_padded_split_replace import digits_for, max_matches, pad

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


def decrypt_indices(ck, out, M, cap):
    from oracle import radix as R
    nd, ni = digits_for(M), digits_for(cap)
    return R.decrypt_radix(ck, out[:nd]), [R.decrypt_radix(ck, out[nd + ni * k: nd + ni * (k + 1)]) for k in range(M)]


CAP = 12
HAYS = [(b"ababa", b"aba"), (b"babababab", b"bab"), (b"a,b,,c,", b","), (b"ab", b""), (b"", b"x"), (b"aaaaaaa", b"aa"),
        (b"xyxyxyz", b"xy"), (b"no match", b"zz")]


def test_match_family_gpu(gpu):
    from oracle import radix as R
    eng, ck, prm = gpu
    M = max_matches(CAP, 0)
    P = Program("pstring_matches", (CAP, 3), params=prm)                          # padded pattern
    for s, pat in HAYS:
        assert R.decrypt_radix(ck, P.run(eng, enc(ck, (s, CAP), (pat, 3)))) == len(rs_match_indices(s, pat)), ("matches", s, pat)
    for op, ref in (("pstring_match_indices", rs_match_indices), ("pstring_rmatch_indices", rs_rmatch_indices)):
        P = Program(op, (CAP, 3), params=prm)
        for s, pat in HAYS:
            want = ref(s, pat)
            assert decrypt_indices(ck, P.run(eng, enc(ck, (s, CAP), (pat, 3))), M, CAP) == (len(want), want + [0] * (M - len(want))), (op, s, pat)
        Mc = max_matches(CAP, 3)
        P = Program(op, (CAP, 3), clear="aba", params=prm)                        # a clear pattern that overlaps itself
        for s in (b"ababababa", b"aba", b"xabaaba"):
            want = ref(s, b"aba")
            assert decrypt_indices(ck, P.run(eng, enc(ck, (s, CAP))), Mc, CAP) == (len(want), want + [0] * (Mc - len(want))), (op, s)
    for op, ref in (("pstring_trim_start_matches", rs_trim_start_matches), ("pstring_trim_end_matches", rs_trim_end_matches)):
        P = Program(op, (CAP, 3), params=prm)
        for s, pat in HAYS:
            assert R.decrypt_string(ck, P.run(eng, enc(ck, (s, CAP), (pat, 3)))) == pad(ref(s, pat), CAP), (op, s, pat)
        P = Program(op, (CAP, 2), clear="ab", params=prm)
        for s in (b"ababxabab", b"abab", b"xab", b"abx"):
            assert R.decrypt_string(ck, P.run(eng, enc(ck, (s, CAP)))) == pad(ref(s, b"ab"), CAP), (op, "clear", s)


def test_lines_and_split_whitespace_gpu(gpu):
    eng, ck, prm = gpu
    P = Program("pstring_lines", (CAP,), params=prm)
    for s in (b"foo\nbar\n\r\nb\r", b"a\n", b"\n", b"", b"\r\r\n", b"one line", b"\n\n\n"):
        assert_split(ck, P.run(eng, enc(ck, (s, CAP))), CAP, CAP, rs_lines(s), ("lines", s))
    P = Program("pstring_split_whitespace", (CAP,), params=prm)
    for s in (b" a\tbc \x0bd\n", b"", b"x\xe3\x80\x80y\xc2\xa0z", b"\xe2\x80\x8bq\xe2\x80\xafr", b"\xe1\x9a\x80\xe2\x81\x9f  ", b"\xc2\x85w\xe2\x80\xa8"):
        assert_split(ck, P.run(eng, enc(ck, (s, CAP))), CAP, (CAP + 1) // 2, rs_split_whitespace(s), ("split_whitespace", s))


# ---- word for word on the coarse lattice ----------------------------------------------------------------------------------------------
EXACT_SPECS = [("pstring_match_indices", (6, 2), None), ("pstring_trim_end_matches", (6, 2), None), ("pstring_lines", (6,), None)]


def test_exact_match_family(orc):
    progs = ExactPrograms(orc, "2_2", 0xF800, EXACT_SPECS)
    eng = progs.engine()
    progs.check(eng, "tuned, fused KS -> PBS", device=True)
    eng.close()


def test_rmatch_indices_sharded_equals_run_device(orc):
    """pstring_rmatch_indices {32, 4} on two ranks of one GPU (DeviceComm.local_group): every rank's words, rounded to the coarse lattice,
    equal program_run_device's"""
    import torch
    import fhe_string_bounty_b200 as F
    from fhe_string_bounty_b200 import multi_gpu as MG
    from helpers import coarse_shift
    p = orc.params("2_2")
    bsk, ksk = coarse_keys(orc, p, 0xF900)
    engines = []
    for _ in range(2):
        e = F.Engine(engine_params(p))
        e.upload_ksk(ksk)
        e.upload_bsk_std(bsk)
        engines.append(e)
    comms = MG.DeviceComm.local_group(engines)
    streams = [torch.cuda.Stream() for _ in comms]
    progs = [Program("pstring_rmatch_indices", (32, 4), params=engine_params(p)) for _ in comms]
    x = coarse_inputs(p, progs[0].n_inputs, 0xF901)
    try:
        def one(r):
            with torch.cuda.stream(streams[r]):
                return comms[r].to_host(MG.run_program_sharded(comms[r], progs[r], x)).copy()
        with ThreadPoolExecutor(2) as pool:
            got = list(pool.map(one, range(2)))
        plan = progs[0].shard_plan(2, comms[0].min_shard_width)
        want = _run_device(engines[0], Program("pstring_rmatch_indices", (32, 4), params=engine_params(p)), x)
    finally:
        for c in comms:
            c.close()
        for e in engines:
            e.close()
    u = coarse_shift(p)
    assert plan[0] > 0, "nothing split"
    assert np.array_equal(got[0], got[1])
    bad = round_to_lattice(got[0], u) != round_to_lattice(want, u)
    print(f"pstring_rmatch_indices(32, 4) at world 2 on one GPU: {plan[0]} split levels, {got[0].size} output words, {int(bad.sum())} differ "
          f"from program_run_device on the 2^{u} lattice; raw words identical: {np.array_equal(got[0], want)}")
    assert not bad.any()


# ---- cost -------------------------------------------------------------------------------------------------------------------------------
def card():
    """name, power limit and max SM clock of device 0 (a read-only query)"""
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        if r.returncode == 0 and r.stdout.strip():
            return r.stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        pass
    import torch
    return torch.cuda.get_device_name(0) + ", power limit unknown"


def test_match_family_cost_gpu(gpu):
    """PBS count, levels and best-of-3 device time at capacity 32"""
    from oracle import radix as R
    eng, ck, prm = gpu
    s = b"ab cd ab ef abab gh ab ijk ab xy"
    ws = b"ab\xe2\x80\x83cd\tef \xe3\x80\x80gh\xc2\xa0ij kl\n"
    M4, Mc = max_matches(32, 0), max_matches(32, 2)
    cases = [("pstring_matches", (32, 4), None, [(s, 32), (b"ab", 4)], lambda out: R.decrypt_radix(ck, out) == s.count(b"ab")),
             ("pstring_match_indices", (32, 2), "ab", [(s, 32)],
              lambda out: decrypt_indices(ck, out, Mc, 32)[1][:s.count(b"ab")] == rs_match_indices(s, b"ab")),
             ("pstring_match_indices", (32, 4), None, [(s, 32), (b"ab", 4)],
              lambda out: decrypt_indices(ck, out, M4, 32)[1][:s.count(b"ab")] == rs_match_indices(s, b"ab")),
             ("pstring_rmatch_indices", (32, 4), None, [(s, 32), (b"ab", 4)],
              lambda out: decrypt_indices(ck, out, M4, 32)[1][:s.count(b"ab")] == rs_rmatch_indices(s, b"ab")),
             ("pstring_trim_start_matches", (32, 4), None, [(b"abababab tail", 32), (b"ab", 4)],
              lambda out: R.decrypt_string(ck, out) == pad(b" tail", 32)),
             ("pstring_trim_end_matches", (32, 4), None, [(b"head xyxyxy", 32), (b"xy", 4)],
              lambda out: R.decrypt_string(ck, out) == pad(b"head ", 32)),
             ("pstring_lines", (32,), None, [(b"one\r\ntwo\n\nthree\nfour\r\n", 32)],
              lambda out: R.decrypt_radix(ck, out[:digits_for(32)]) == len(rs_lines(b"one\r\ntwo\n\nthree\nfour\r\n"))),
             ("pstring_split_whitespace", (32,), None, [(ws, 32)], lambda out: R.decrypt_radix(ck, out[:digits_for(16)]) == len(rs_split_whitespace(ws)))]
    print(f"\n# {card()}")
    for op, args, clear, strings, ok in cases:
        P = Program(op, args, clear=clear, params=prm)
        x = enc(ck, *strings)
        out = P.run(eng, x)
        assert ok(out), (op, args, clear)
        ms = []
        for _ in range(3):
            P.run(eng, x)
            ms.append(P.last_ms())
        print(f"{op}{args}{', clear ' + repr(clear) if clear else ''}: {P.n_pbs} PBS in {P.n_levels} levels, "
              f"device {min(ms):.1f} ms (best of 3; {', '.join(f'{m:.1f}' for m in ms)})")
