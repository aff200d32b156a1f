"""Any recorded program across several ranks (run with -m gpu): multi_gpu.run_program_sharded / tfhe_b200_program_run_sharded[_group].

Levels wider than min_shard_width are split across the ranks and put back into every rank's arena by the scatter exchange
(csrc/exchange.cu); the others run in full on every rank.  On one GPU the ranks are a DeviceComm.local_group (one cooperative scatter per
split level).  The word-for-word checks reuse the coarse lattice of tests/test_gpu_exact_programs.py: every rank's outputs rounded to 2^u
must equal the exact executor, and all ranks must hold the same raw words (every split row is computed once and copied)."""
import ctypes as C
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from fhe_string_bounty_b200.host import Program
from helpers import engine_params, max_coef_sum, max_residual, round_to_lattice
from test_gpu_exact_programs import PROGRAMS_2_2, SEED_2_2, ExactPrograms, _run_device, assert_residual

pytestmark = pytest.mark.gpu


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def progs_2_2(orc):
    return ExactPrograms(orc, "2_2", SEED_2_2, PROGRAMS_2_2)


class Group:
    """`world` ranks on one GPU: one engine (same coarse keys), comm, stream and Program object per rank"""

    def __init__(self, progs, world, min_shard_width):
        import torch
        from fhe_string_bounty_b200 import multi_gpu as MG
        self.progs, self.world = progs, world
        self.engines = [progs.engine() for _ in range(world)]
        self.comms = MG.DeviceComm.local_group(self.engines)
        for c in self.comms:
            c.min_shard_width = min_shard_width
        self.streams = [torch.cuda.Stream() for _ in self.comms]
        self.programs = {}

    def program(self, r, case):
        key = (r, case["label"])
        if key not in self.programs:
            op, args, clear = case["spec"]
            self.programs[key] = Program(op, args, clear=clear, params=engine_params(self.progs.p))
        return self.programs[key]

    def all_ranks(self, fn):
        import torch

        def one(r):
            with torch.cuda.stream(self.streams[r]):
                return fn(r, self.comms[r])
        with ThreadPoolExecutor(self.world) as pool:
            return list(pool.map(one, range(self.world)))

    def run(self, case):
        from fhe_string_bounty_b200 import multi_gpu as MG
        return self.all_ranks(lambda r, c: c.to_host(MG.run_program_sharded(c, self.program(r, case), case["ins"])).copy())

    def close(self):
        for P in self.programs.values():
            P.close()
        for c in self.comms:
            c.close()
        for e in self.engines:
            e.close()


def _cases(progs, specs):
    by_label = {c["label"]: c for c in progs.cases}
    out = []
    for op, args, clear in specs:
        c = by_label[f"{op}{args}" + (f" clear {clear!r}" if clear else "")]
        out.append(dict(c, spec=(op, args, clear)))
    return out


def check_group(progs, world, min_shard_width, specs):
    g = Group(progs, world, min_shard_width)
    worst, coef, n_split = 0, world, 0
    try:
        for case in _cases(progs, specs):
            got = g.run(case)
            plan = case["P"].shard_plan(world, min_shard_width)
            n_split += plan[0]
            for r in range(world):
                assert np.array_equal(got[r], got[0]), f"{case['label']}: rank {r} holds other words than rank 0"
                bad = round_to_lattice(got[r], progs.u) != case["exact"]
                assert not bad.any(), (f"[{progs.name}] {case['label']}, world {world}, min_shard_width {min_shard_width}, rank {r} "
                                       f"(plan {plan}): {int(bad.sum())} words in rows {np.flatnonzero(bad.any(axis=1))[:8].tolist()}")
            worst = max(worst, max_residual(got[0], case["exact"]))
            coef = max(coef, max_coef_sum(case["ir"]))
    finally:
        g.close()
    assert_residual(progs.p, f"[{progs.name}] sharded programs, world {world}, min_shard_width {min_shard_width}: {len(specs)} programs, "
                    f"{n_split} split levels", worst, coef)
    return n_split


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("min_w", ["0", "sms"])
def test_2_2_sharded_exact(progs_2_2, world, min_w):
    """min_shard_width 0 splits every level, the narrow ones into empty shares and widths not divisible by world; SM count mixes split
    and replicated levels"""
    m = 0 if min_w == "0" else _sms()
    n_split = check_group(progs_2_2, world, m, PROGRAMS_2_2)
    assert n_split > 0
    if m == 0:      # levels narrower than `world` are split too: some ranks run empty shares
        assert any(w < world for c in progs_2_2.cases for w in c["ir"].level_widths)


OTHER = {"multibit_2_2_g3": [("string_contains", (12, 3), None)], "1_1": [("string_eq", (20, 20), None)],
         "2_3": [("string_contains", (4, 2), None)]}


@pytest.mark.parametrize("name", list(OTHER))
def test_other_kernel_families_sharded(orc, name):
    progs = ExactPrograms(orc, name, 0xF500, OTHER[name])
    assert check_group(progs, 2, 0, OTHER[name]) > 0


def test_nothing_split_equals_run_device(progs_2_2):
    """min_shard_width above every width: the same kernels as program_run_device, so the same words"""
    m = max(w for c in progs_2_2.cases for w in c["ir"].level_widths)
    g = Group(progs_2_2, 2, m)
    try:
        for case in _cases(progs_2_2, PROGRAMS_2_2):
            assert case["P"].shard_plan(2, m)[0] == 0
            got = g.run(case)
            want = _run_device(g.engines[0], g.program(0, case), case["ins"])
            for r in range(2):
                assert np.array_equal(got[r], want), f"{case['label']}, rank {r}"
    finally:
        g.close()


def test_epochs_interleave_with_sharded_contains(progs_2_2):
    """program, multi_gpu.sharded_contains on the same comms (the 16-row peer exchange), then the program again: every result is the
    one the comms computed before any other exchange ran"""
    from fhe_string_bounty_b200 import multi_gpu as MG
    from test_gpu_exact_programs import _sharded_inputs
    case = _cases(progs_2_2, [("pstring_split", (8, 2), None)])[0]
    g = Group(progs_2_2, 2, 0)
    try:
        x = _sharded_inputs(progs_2_2.p)
        prm = engine_params(progs_2_2.p)
        contains = lambda: g.all_ranks(lambda r, c: MG.sharded_contains(c, prm, x["hay"], x["pat"], 12, 3))
        contains0 = contains()
        first = g.run(case)
        contains1 = contains()
        again = g.run(case)
    finally:
        g.close()
    for r in range(2):
        assert np.array_equal(round_to_lattice(first[r], progs_2_2.u), case["exact"])
        assert np.array_equal(again[r], first[r])
        assert np.array_equal(contains1[r], contains0[r])


# ---- real keys, world 2 on one GPU: decrypted against Python bytes ---------------------------------------------------------------------

@pytest.fixture(scope="module")
def real_group(keys_2_2):
    import torch
    import fhe_string_bounty_b200 as F
    from fhe_string_bounty_b200 import multi_gpu as MG
    p, ck, sk = keys_2_2
    engines = []
    for _ in range(2):
        e = F.Engine(engine_params(p))
        e.upload_ksk(sk.ksk)
        e.upload_bsk_std(sk.bsk)
        engines.append(e)
    comms = MG.DeviceComm.local_group(engines)
    streams = [torch.cuda.Stream() for _ in comms]

    def run(op, args, clear, x):
        progs = [Program(op, args, clear=clear, params=engine_params(p)) for _ in comms]

        def one(r):
            with torch.cuda.stream(streams[r]):
                return comms[r].to_host(MG.run_program_sharded(comms[r], progs[r], x)).copy()
        with ThreadPoolExecutor(2) as pool:
            outs = list(pool.map(one, range(2)))
        assert progs[0].shard_plan(2, comms[0].min_shard_width)[0] > 0, f"{op}{args}: nothing split"
        assert np.array_equal(outs[0], outs[1])
        return outs[0]
    yield run, ck
    for c in comms:
        c.close()
    for e in engines:
        e.close()


def test_real_keys_split_replace(real_group):
    from oracle import radix as R
    from test_padded_split_replace import digits_for, max_matches, pad, rs_replacen, rs_splitn
    run, ck = real_group
    enc = lambda *strings: np.concatenate([R.encrypt_string(ck, pad(s, c)) for s, c in strings])
    s = b"ab cd ab ef abab gh ab ijk ab xy"
    out = run("pstring_split", (32, 4), None, enc((s, 32), (b"ab", 4)))
    Pn = max_matches(32, 0) + 1
    nd = digits_for(Pn)
    want = rs_splitn(s, b"ab", None)
    assert R.decrypt_radix(ck, out[:nd]) == len(want)
    parts = [R.decrypt_string(ck, out[nd + 4 * 32 * k: nd + 4 * 32 * (k + 1)]) for k in range(Pn)]
    assert parts == [pad(w, 32) for w in want] + [pad(b"", 32)] * (Pn - len(want))
    out = run("pstring_replace", (32, 4, 4), None, enc((s, 32), (b"ab", 4), (b"XY!", 4)))
    assert R.decrypt_string(ck, out) == pad(rs_replacen(s, b"ab", b"XY!"), 32 + max_matches(32, 0) * 4)


def test_real_keys_eq_many(real_group):
    from oracle import radix as R
    run, ck = real_group
    pairs = [(b"abcdefgh", b"abcdefgh"), (b"abcdefgh", b"abcdefgX"), (b"zzzzzzzz", b"zzzzzzzz"), (b"\x00\x01\x02\x03\x04\x05\x06\x07", b"01234567")] * 16
    x = np.concatenate([R.encrypt_string(ck, s) for a, b in pairs for s in (a, b)])
    out = run("string_eq_many", (8, 8, len(pairs)), None, x)
    assert [ck.decrypt_message_and_carry(o) for o in out] == [int(a == b) for a, b in pairs]


# ---- errors: refused before anything is enqueued ---------------------------------------------------------------------------------------

def test_errors_enqueue_nothing(progs_2_2):
    import torch
    from fhe_string_bounty_b200._native import NativeError
    from fhe_string_bounty_b200 import multi_gpu as MG
    case = _cases(progs_2_2, [("string_contains", (96, 8), None)])[0]
    g = Group(progs_2_2, 2, 0)
    lib = g.engines[0].lib
    try:
        P = [g.program(r, case) for r in range(2)]
        need = P[0].shard_plan(2, 0)[1]
        small = [MG.PeerExchange.local(g.engines[r], r, 2, need - 1) for r in range(2)]
        arr = (C.c_void_p * 2)(*[x.h for x in small])
        for x in small:
            g.engines[0]._check(lib.tfhe_b200_exchange_attach_local(x.h, arr))
        ins = torch.from_numpy(case["ins"].view(np.int64)).cuda()
        outs = [torch.empty((P[0].n_outputs, g.comms[0].L), dtype=torch.int64, device="cuda") for _ in range(2)]
        ptrs = lambda xs: (C.c_void_p * 2)(*xs)

        def group_call(ctxs, progs, exs):
            rc = lib.tfhe_b200_program_run_sharded_group(ptrs(ctxs), ptrs(progs), ptrs(exs), 2, ptrs([ins.data_ptr()] * 2),
                                                         ptrs([o.data_ptr() for o in outs]), 0, None)
            assert rc != 0
            return lib.tfhe_b200_last_error().decode()

        ctxs, progs = [e.h for e in g.engines], [p.h for p in P]
        launches = [e.kernel_launches for e in g.engines]
        msg = group_call(ctxs, progs, [x.h for x in small])
        assert f"max_rows >= {need}" in msg, msg
        msg = group_call(ctxs[::-1], progs, [x.h for x in small])        # rank 0's exchange with rank 1's context
        assert "belongs to another context" in msg, msg
        other = Program("string_contains", (96, 8), params=dict(engine_params(progs_2_2.p), msg_mod=2, carry_mod=8))
        msg = group_call(ctxs, [other.h, P[1].h], [x.h for x in small])
        assert "other parameters" in msg, msg
        # nothing split (so the exchange is large enough), but both ranks live on this GPU
        rc = lib.tfhe_b200_program_run_sharded(ctxs[0], progs[0], small[0].h, ins.data_ptr(), outs[0].data_ptr(), 1 << 40, None)
        assert rc != 0 and "share a GPU" in lib.tfhe_b200_last_error().decode()
        assert [e.kernel_launches for e in g.engines] == launches, "a refused call enqueued work"
        for x in small:
            x.close()
        other.close()
        with pytest.raises(ValueError, match="nccl"):
            MG.run_program_sharded(MG.DeviceComm(g.engines[0], rank=0, world=2, exchange="nccl"), P[0], case["ins"])
        got = g.run(case)                         # a normal run afterwards
        for r in range(2):
            assert np.array_equal(round_to_lattice(got[r], progs_2_2.u), case["exact"])
    finally:
        g.close()


@pytest.mark.skipif("not __import__('torch').cuda.is_available() or __import__('torch').cuda.device_count() < 2",
                    reason="needs two GPUs")
def test_two_gpus_run_sharded(progs_2_2):
    """world 2 across two devices through tfhe_b200_program_run_sharded (one rank per GPU, driven from two threads), and a group across
    the two devices is refused"""
    import torch
    import fhe_string_bounty_b200 as F
    from fhe_string_bounty_b200 import multi_gpu as MG
    from helpers import engine_params as ep
    case = _cases(progs_2_2, [("pstring_split", (8, 2), None)])[0]
    engines = []
    for d in range(2):
        e = F.Engine(ep(progs_2_2.p), device=d)
        e.upload_ksk(progs_2_2.ksk)
        e.upload_bsk_std(progs_2_2.bsk)
        engines.append(e)
    lib = engines[0].lib
    P = [Program(*case["spec"][:2], clear=case["spec"][2], params=ep(progs_2_2.p)) for _ in range(2)]
    need = max(1, P[0].shard_plan(2, 0)[1])
    exs = [MG.PeerExchange.local(engines[r], r, 2, need) for r in range(2)]
    arr = (C.c_void_p * 2)(*[x.h for x in exs])
    for r in range(2):
        engines[r]._check(lib.tfhe_b200_exchange_attach_local(exs[r].h, arr))
    ins = [torch.from_numpy(case["ins"].view(np.int64)).to(f"cuda:{d}") for d in range(2)]
    outs = [torch.empty((P[0].n_outputs, progs_2_2.p.glwe_dim * progs_2_2.p.poly_size + 1), dtype=torch.int64, device=f"cuda:{d}")
            for d in range(2)]
    ptrs = lambda xs: (C.c_void_p * 2)(*xs)
    rc = lib.tfhe_b200_program_run_sharded_group(ptrs([e.h for e in engines]), ptrs([p.h for p in P]), ptrs([x.h for x in exs]), 2,
                                                 ptrs([t.data_ptr() for t in ins]), ptrs([o.data_ptr() for o in outs]), 0, None)
    assert rc != 0 and "a group runs on one GPU" in lib.tfhe_b200_last_error().decode()

    def one(r):
        with torch.cuda.device(r):
            s = torch.cuda.Stream()
            engines[r]._check(lib.tfhe_b200_program_run_sharded(engines[r].h, P[r].h, exs[r].h, ins[r].data_ptr(), outs[r].data_ptr(), 0,
                                                                s.cuda_stream))
            s.synchronize()
            return outs[r].cpu().numpy().view(np.uint64).copy()
    with ThreadPoolExecutor(2) as pool:
        got = list(pool.map(one, range(2)))
    for x in exs:
        x.close()
    for p in P:
        p.close()
    for e in engines:
        e.close()
    assert np.array_equal(got[0], got[1])
    assert np.array_equal(round_to_lattice(got[0], progs_2_2.u), case["exact"])
