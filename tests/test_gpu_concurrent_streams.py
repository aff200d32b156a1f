"""Calls in flight at the same time on one context, on several streams (run with -m gpu).

The device entry points take any stream, and the context's mutex only orders the enqueues: the kernels of one call can still run when
the next call is enqueued on another stream.  Calls of one context share its keyswitch digit buffer and its keyswitch -> PBS hand-off
rows, and runs of one program share the program's arena; the context orders them with events (tbc::StreamOrder).  Here the calls of a
schedule are all enqueued before anything is synchronised, each stream with its own inputs, LUT indices and batch size, from one thread
or from one thread per stream, and every output is compared word for word with an exact reference:
  * keyswitch_batch_device on every keyswitch kernel, two and three streams (one of them the context's own stream), against
    orc_keyswitch on every row;
  * ks_pbs_batch_device and ks_pbs_many_batch_device (real KSK, lattice BSK as in test_gpu_exact_rotation.py): probe rows (first, middle
    and last CTAs) rounded to 2^s against the exact rotation of the oracle keyswitch, every row against the same call run alone on the
    same context; a wide level (v4 + v8 tail) beside a narrow one (v8x2), fused and unfused hand-off;
  * pbs_batch_device on the generic kernel (N = 4096) and its launch_big path (N = 16384), whose scratch is stream-ordered;
  * programs on the coarse lattice of test_gpu_exact_programs.py against run_program_exact: two programs, one program twice (its arena),
    and Program.run on the host entry while a program_run_device call is pending;
  * the host entries keyswitch_batch and pbs_ks_batch while a multi-wave ks_pbs_batch_device call is pending.
"presized" schedules run after the same calls ran alone, so no buffer grows; "growth" schedules start on a fresh context with the
smallest call, so the shared buffers grow while it is pending.  A mismatch names the stream, the row and whether the wrong row equals a
row expected from another call of the schedule ("crossed": shared scratch) or none ("garbage").
"""
import threading

import numpy as np
import pytest

from helpers import (engine_params, exact_unique, keyswitch_rows, lattice_bsk, lattice_inputs, lattice_luts, lattice_shift,
                     max_coef_sum, max_residual, round_to_lattice)
from many_lut_ref import exact_glwe_batch, extract_at, extraction_step
from test_gpu_exact_programs import SEED_2_2, ExactPrograms, assert_residual

pytestmark = pytest.mark.gpu


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint64).view(np.int64)).cuda()


def _zeros(*shape):
    import torch
    return torch.zeros(int(np.prod(shape)), dtype=torch.int64, device="cuda")


def _host(t, *shape):
    return t.cpu().numpy().view(np.uint64).reshape(shape)


def _engine(p, ksk=None, bsk=None, tuning=None):
    import fhe_string_bounty_b200 as F
    e = F.Engine(engine_params(p))
    for k, v in (tuning or {}).items():      # ks_kernel before the KSK upload
        e.set_tuning(k, v)
    if ksk is not None:
        e.upload_ksk(ksk)
    if bsk is not None:
        e.upload_bsk_std(bsk)
    return e


def _probe_rows(batch, sms):
    """first and last CTAs, the middle, and the rows around the end of the first wide wave"""
    rows = {0, 1, 2, 3, batch // 2, batch - 3, batch - 2, batch - 1, 4 * sms - 1, 4 * sms}
    return sorted(r for r in rows if 0 <= r < batch)


def run_schedule(calls, threads):
    """calls: [(stream, enqueue)], enqueue(handle) enqueues one call on that stream handle (None: the context's stream).  One thread in
    list order, or one thread per call started together; nothing is synchronised before every call is enqueued."""
    import torch
    torch.cuda.synchronize()             # the inputs, copied on the current stream, are in place
    if not threads:
        for s, enqueue in calls:
            enqueue(s.cuda_stream if s is not None else None)
    else:
        go, errors = threading.Barrier(len(calls)), []

        def one(s, enqueue):
            try:
                go.wait()
                if s is None:
                    enqueue(None)
                else:
                    with torch.cuda.stream(s):
                        enqueue(s.cuda_stream)
            except BaseException as e:      # re-raised below, in the test's thread
                errors.append(e)
        ts = [threading.Thread(target=one, args=c) for c in calls]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        if errors:
            raise errors[0]
    torch.cuda.synchronize()


class Report:
    """word-for-word comparisons of one schedule; every call is checked before the test fails, so the report counts all wrong words"""

    def __init__(self, label):
        self.label, self.words, self.lines, self.checked = label, 0, [], 0

    def compare(self, call, got, want, others, what="words"):
        """got / want: (rows, words); others: {call name: rows expected from the other calls of the schedule}"""
        got, want = got.reshape(len(got), -1), want.reshape(len(want), -1)
        bad = got != want
        self.checked += bad.size
        if not bad.any():
            return
        self.words += int(bad.sum())
        rows = np.flatnonzero(bad.any(axis=1))
        index = {}      # whole rows, and mask words alone (a keyswitch that read another call's digits keeps its own body)
        for name, o in others.items():
            for j, r in enumerate(o.reshape(len(o), -1)):
                index.setdefault(r.tobytes(), f"crossed: equals row {j} of {name}")
                index.setdefault(r[:-1].tobytes(), f"crossed: mask words equal row {j} of {name}")
        where = [f"row {int(r)}: {int(bad[r].sum())} words, "
                 f"{index.get(got[r].tobytes(), index.get(got[r][:-1].tobytes(), 'garbage'))}" for r in rows[:6]]
        self.lines.append(f"{call}: {int(bad.sum())} wrong {what} in {len(rows)} of {len(got)} rows; " + "; ".join(where))

    def done(self):
        print(f"{self.label}: {self.words} mismatching words of {self.checked} compared")
        assert not self.lines, f"{self.label}: {self.words} mismatching words\n  " + "\n  ".join(self.lines)


MODES = [False, True]
MODE_IDS = ["same_thread", "two_threads"]


# ---- keyswitch_batch_device ---------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ks_sets(orc, keys_2_2):
    """three input sets of distinct random big LWEs: 64 * SMs (many waves), SMs + 3 and 2 * SMs + 5 rows, with orc_keyswitch of every row"""
    p, ck, sk = keys_2_2
    sms = _sms()
    out = []
    for i, rows in enumerate((64 * sms, sms + 3, 2 * sms + 5)):
        big = np.random.default_rng(0xC000 + i).integers(0, 2**64, size=(rows, p.big_dim + 1), dtype=np.uint64)
        out.append((big, keyswitch_rows(orc, p, sk.ksk, big)))
    return out


@pytest.mark.parametrize("threads", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("growth", [False, True], ids=["presized", "growth"])
@pytest.mark.parametrize("n_streams", [2, 3])
@pytest.mark.parametrize("ks_kernel", [2, 1, 0])
def test_keyswitch_streams(keys_2_2, ks_sets, ks_kernel, n_streams, growth, threads):
    import torch
    p, ck, sk = keys_2_2
    eng = _engine(p, ksk=sk.ksk, tuning={"ks_kernel": ks_kernel})
    sets = ks_sets[:n_streams]
    d_in = [_dev(big) for big, _ in sets]
    d_out = [_zeros(len(big), p.lwe_dim + 1) for big, _ in sets]
    # the third call goes to the context's own stream (handle NULL)
    streams = [torch.cuda.Stream(), torch.cuda.Stream(), None][:n_streams]
    if not growth:
        for i in range(n_streams):        # alone first: the digit buffer reaches its largest size before the schedule
            eng.keyswitch_batch_device(d_in[i], d_out[i], len(sets[i][0]), streams[i].cuda_stream if streams[i] else None)
        torch.cuda.synchronize()
        for t in d_out:
            t.zero_()
    order = sorted(range(n_streams), key=lambda i: len(sets[i][0])) if growth else list(range(n_streams))
    run_schedule([(streams[i], lambda h, i=i: eng.keyswitch_batch_device(d_in[i], d_out[i], len(sets[i][0]), h)) for i in order], threads)
    rep = Report(f"keyswitch_batch_device, ks_kernel {ks_kernel}, {n_streams} streams, {'growth' if growth else 'no growth'}, "
                 f"{MODE_IDS[threads]}")
    for i in range(n_streams):
        others = {f"stream {j}": sets[j][1] for j in range(n_streams) if j != i}
        rep.compare(f"stream {i} (batch {len(sets[i][0])})", _host(d_out[i], len(sets[i][0]), p.lwe_dim + 1), sets[i][1], others)
    eng.close()
    rep.done()


# ---- ks_pbs_batch_device and ks_pbs_many_batch_device -----------------------------------------------------------------------------

class KsPbsCase:
    """real 2_2 KSK, lattice BSK and LUTs; per stream: fresh encryptions, LUT indices, probe rows and their exact outputs"""

    def __init__(self, orc, keys, sms):
        self.orc = orc
        self.p, self.ck, self.sk = keys
        p = self.p
        self.s = lattice_shift(p)
        self.bsk = lattice_bsk(orc, p, 0xC100)
        self.luts = lattice_luts(p, 3, 0xC101)
        self.fcounts = np.array([2, 3, 4], dtype=np.uint32)
        self.streams = []
        for i, (rows, step) in enumerate(((4 * sms + 3, 7), (sms // 2, 5), (12 * sms + 1, 2))):
            rng = np.random.default_rng(0xC200 + i)
            cts = self.ck.encrypt_batch(rng.integers(0, 16, size=rows))
            idx = ((np.arange(rows) * step + i) % len(self.luts)).astype(np.uint32)
            probe = _probe_rows(rows, sms)
            small = np.stack([self.sk.keyswitch(cts[r]) for r in probe])
            self.streams.append(dict(cts=cts, idx=idx, probe=probe, small=small,
                                     exact=exact_unique(orc, p, self.bsk, small, self.luts, idx[probe])))

    def many_exact(self, i):
        """(probe row, function) pairs of call i and the extraction at t_f of the exact GLWE of each"""
        c, p = self.streams[i], self.p
        g = exact_glwe_batch(p, self.bsk, c["small"], self.luts, c["idx"][c["probe"]])
        pairs, rows = [], []
        for k, r in enumerate(c["probe"]):
            F = int(self.fcounts[c["idx"][r]])
            for f in range(F):
                pairs.append((r, f))
                rows.append(extract_at(g[k][None], f * extraction_step(p, F))[0])
        return pairs, np.stack(rows)


@pytest.fixture(scope="module")
def kspbs(orc, keys_2_2):
    return KsPbsCase(orc, keys_2_2, _sms())


def _kspbs_schedule(case, eng, calls, growth, threads, many):
    """calls: indices into case.streams, in enqueue order, one stream each.  Returns (got, solo) per call, solo = the call run alone on
    the same context (before the schedule, or after it for a growth schedule, whose point is a context that has not run yet)"""
    import torch
    p, L = case.p, case.p.big_dim + 1
    S = int(case.fcounts.max()) if many else 1
    fn = eng.ks_pbs_many_batch_device if many else eng.ks_pbs_batch_device
    d_in = {i: _dev(case.streams[i]["cts"]) for i in calls}
    d_idx = {i: torch.from_numpy(case.streams[i]["idx"].view(np.int32)).cuda() for i in calls}
    d_out = {i: _zeros(len(case.streams[i]["cts"]), S, L) for i in calls}
    streams = {i: torch.cuda.Stream() for i in calls}

    def alone():
        res = {}
        for i in calls:
            d_out[i].zero_()
            torch.cuda.synchronize()
            fn(d_in[i], d_idx[i], d_out[i], len(case.streams[i]["cts"]), streams[i].cuda_stream)
            torch.cuda.synchronize()
            res[i] = _host(d_out[i], len(case.streams[i]["cts"]), S, L).copy()
            d_out[i].zero_()
        return res
    solo = None if growth else alone()
    run_schedule([(streams[i], lambda h, i=i: fn(d_in[i], d_idx[i], d_out[i], len(case.streams[i]["cts"]), h)) for i in calls], threads)
    got = {i: _host(d_out[i], len(case.streams[i]["cts"]), S, L).copy() for i in calls}
    if growth:
        solo = alone()
    return got, solo


def _check_kspbs(case, rep, got, solo, many):
    p, s = case.p, case.s
    for i in got:
        c = case.streams[i]
        name = f"stream of batch {len(c['cts'])}"
        others = {f"batch {len(case.streams[j]['cts'])}": solo[j] for j in got if j != i}
        rep.compare(f"{name}, every row == the call alone", got[i], solo[i], others)
        if many:
            pairs, exact = case.many_exact(i)
            rows = np.stack([got[i][r, f] for r, f in pairs])
        else:
            rows, exact = got[i][c["probe"]], c["exact"]
        rep.compare(f"{name}, probe rows {c['probe']} rounded to 2^{s} == exact", round_to_lattice(rows, s), exact, {}, "lattice words")


KSPBS_PAIRS = [("wide v4 + v8 tail, narrow v8x2", {}, (0, 1)), ("unfused hand-off (ks_kernel 0)", {"ks_kernel": 0}, (0, 1))]


@pytest.mark.parametrize("threads", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("growth", [False, True], ids=["presized", "growth"])
@pytest.mark.parametrize("pair", KSPBS_PAIRS, ids=["fused", "unfused"])
def test_ks_pbs_streams(kspbs, pair, growth, threads):
    label, tuning, calls = pair
    eng = _engine(kspbs.p, ksk=kspbs.sk.ksk, bsk=kspbs.bsk, tuning=tuning)
    eng.upload_luts(kspbs.luts)
    order = sorted(calls, key=lambda i: len(kspbs.streams[i]["cts"])) if growth else list(calls)
    got, solo = _kspbs_schedule(kspbs, eng, order, growth, threads, many=False)
    eng.close()
    rep = Report(f"ks_pbs_batch_device, {label}, {'growth' if growth else 'no growth'}, {MODE_IDS[threads]}")
    _check_kspbs(kspbs, rep, got, solo, many=False)
    rep.done()


@pytest.mark.parametrize("threads", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("growth", [False, True], ids=["presized", "growth"])
def test_ks_pbs_many_streams(kspbs, growth, threads):
    eng = _engine(kspbs.p, ksk=kspbs.sk.ksk, bsk=kspbs.bsk)
    eng.upload_many_luts(kspbs.luts, kspbs.fcounts)
    order = [1, 0] if growth else [0, 1]
    got, solo = _kspbs_schedule(kspbs, eng, order, growth, threads, many=True)
    eng.close()
    rep = Report(f"ks_pbs_many_batch_device, F in {kspbs.fcounts.tolist()}, {'growth' if growth else 'no growth'}, {MODE_IDS[threads]}")
    _check_kspbs(kspbs, rep, got, solo, many=True)
    rep.done()


def test_host_entries_during_pending_device_call(kspbs, keys_2_2):
    """ks_pbs_batch_device of 12 * SMs + 1 rows (several waves) on stream A, then keyswitch_batch and pbs_ks_batch on the context's stream
    without synchronising A: keyswitch_batch against orc_keyswitch, the other two against the same calls alone"""
    import torch
    case, (p, ck, sk) = kspbs, keys_2_2
    a = case.streams[2]
    batch = len(a["cts"])
    eng = _engine(p, ksk=sk.ksk, bsk=case.bsk)
    eng.upload_luts(case.luts)
    ks_in = case.streams[0]["cts"]
    ks_want = keyswitch_rows(case.orc, p, sk.ksk, ks_in)
    pk_in = lattice_inputs(p, 3 * _sms() + 1, 0xC300)
    pk_idx = (np.arange(len(pk_in)) % len(case.luts)).astype(np.uint32)
    d_in, d_idx, d_out = _dev(a["cts"]), torch.from_numpy(a["idx"].view(np.int32)).cuda(), _zeros(batch, p.big_dim + 1)
    sA = torch.cuda.Stream()
    # alone first (every shared buffer at its final size): the references of the device call and of pbs_ks_batch
    eng.ks_pbs_batch_device(d_in, d_idx, d_out, batch, sA.cuda_stream)
    torch.cuda.synchronize()
    solo = _host(d_out, batch, p.big_dim + 1).copy()
    pk_solo = eng.pbs_ks_batch(pk_in, pk_idx)
    assert np.array_equal(eng.keyswitch_batch(ks_in), ks_want)
    d_out.zero_()
    torch.cuda.synchronize()
    eng.ks_pbs_batch_device(d_in, d_idx, d_out, batch, sA.cuda_stream)
    ks_got = eng.keyswitch_batch(ks_in)
    pk_got = eng.pbs_ks_batch(pk_in, pk_idx)
    torch.cuda.synchronize()
    got = _host(d_out, batch, p.big_dim + 1)
    eng.close()
    rep = Report("host entries while ks_pbs_batch_device is pending")
    rep.compare("ks_pbs_batch_device, every row == alone", got, solo, {})
    rep.compare(f"ks_pbs_batch_device, probe rows rounded to 2^{case.s} == exact", round_to_lattice(got[a["probe"]], case.s), a["exact"], {},
                "lattice words")
    rep.compare("keyswitch_batch == orc_keyswitch", ks_got, ks_want, {})
    rep.compare("pbs_ks_batch == alone", pk_got, pk_solo, {})
    rep.done()


# ---- pbs_batch_device on the generic kernel ---------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["2_3", "4_3"])
def test_generic_pbs_streams(orc, name):
    """2_3: pbs_generic_kernel (N = 4096); 4_3: launch_big (N = 16384, two levels), whose grid-stride scratch is allocated on the call's
    stream"""
    import torch
    p = orc.params(name)
    s, sms = lattice_shift(p), _sms()
    bsk, luts = lattice_bsk(orc, p, 0xC400), lattice_luts(p, 3, 0xC401)
    sizes = (2 * sms + 5, 7) if p.poly_size > 4096 else (3 * sms + 1, 24)
    n_probe = 3 if p.poly_size > 4096 else 8
    calls = []
    for i, rows in enumerate(sizes):
        small = lattice_inputs(p, rows, 0xC410 + i)
        idx = ((np.arange(rows) * (i + 2) + i) % len(luts)).astype(np.uint32)
        probe = sorted({0, rows // 2, rows - 1} | set(range(min(rows, n_probe - 3))))
        calls.append(dict(small=small, idx=idx, probe=probe, exact=exact_unique(orc, p, bsk, small[probe], luts, idx[probe])))
    eng = _engine(p, bsk=bsk)
    eng.upload_luts(luts)
    L = p.big_dim + 1
    for c in calls:
        c["d_in"], c["d_idx"], c["d_out"] = _dev(c["small"]), torch.from_numpy(c["idx"].view(np.int32)).cuda(), _zeros(len(c["small"]), L)
        c["stream"] = torch.cuda.Stream()
    for c in calls:
        eng.pbs_batch_device(c["d_in"], c["d_idx"], c["d_out"], len(c["small"]), c["stream"].cuda_stream)
        torch.cuda.synchronize()
        c["solo"] = _host(c["d_out"], len(c["small"]), L).copy()
        c["d_out"].zero_()
    run_schedule([(c["stream"], lambda h, c=c: eng.pbs_batch_device(c["d_in"], c["d_idx"], c["d_out"], len(c["small"]), h)) for c in calls],
                 False)
    eng.close()
    rep = Report(f"pbs_batch_device [{name}], batches {sizes}")
    for i, c in enumerate(calls):
        got = _host(c["d_out"], len(c["small"]), L)
        rep.compare(f"stream {i}, every row == alone", got, c["solo"], {f"stream {j}": calls[j]["solo"] for j in range(len(calls)) if j != i})
        rep.compare(f"stream {i}, probe rows {c['probe']} rounded to 2^{s} == exact", round_to_lattice(got[c["probe"]], s), c["exact"], {},
                    "lattice words")
    rep.done()


# ---- programs -----------------------------------------------------------------------------------------------------------------------

PROGRAM_SPECS = [("string_contains", (32, 4), None), ("pstring_split", (8, 2), None), ("pstring_split", (8, 2), None)]


@pytest.fixture(scope="module")
def progs(orc):
    """the coarse 2_2 lattice; cases 1 and 2 are the same program with different inputs"""
    return ExactPrograms(orc, "2_2", SEED_2_2 + 0x40, PROGRAM_SPECS)


def _run_device(eng, P, d_in, d_out, handle):
    eng._check(eng.lib.tfhe_b200_program_run_device(eng.h, P.h, d_in.data_ptr(), d_out.data_ptr(), handle))


def _program_schedule(progs, runs, threads, host=None):
    """runs: [(program case, input case)] on streams of their own, through program_run_device; host: a (program case, input case) run
    through Program.run on the host entry after the device runs are enqueued.  Returns (got per run, host output)"""
    import torch
    eng = progs.engine()
    for c in progs.cases:                # alone first: binds the programs, and d_small and the digits reach their final sizes
        c["P"].run(eng, c["ins"])
    L = progs.p.big_dim + 1
    d_in = [_dev(progs.cases[ic]["ins"]) for _, ic in runs]
    d_out = [_zeros(progs.cases[ic]["P"].n_outputs, L) for _, ic in runs]
    streams = [torch.cuda.Stream() for _ in runs]
    calls = [(streams[k], lambda h, k=k: _run_device(eng, progs.cases[runs[k][0]]["P"], d_in[k], d_out[k], h)) for k in range(len(runs))]
    host_out = None
    if host is None:
        run_schedule(calls, threads)
    else:
        torch.cuda.synchronize()
        for s, enqueue in calls:
            enqueue(s.cuda_stream)
        host_out = progs.cases[host[0]]["P"].run(eng, progs.cases[host[1]]["ins"])
        torch.cuda.synchronize()
    got = [_host(d_out[k], progs.cases[runs[k][0]]["P"].n_outputs, L) for k in range(len(runs))]
    eng.close()
    return got, host_out


def _check_programs(progs, rep, outs):
    """outs: [(label, input case, output rows)]: rounded to 2^u == the exact executor's, every word"""
    worst, coef = 0, 1
    for label, ic, got in outs:
        want = progs.cases[ic]["exact"]
        others = {f"{progs.cases[j]['label']} inputs {j}": progs.cases[j]["exact"] for j in range(len(progs.cases))
                  if j != ic and progs.cases[j]["exact"].shape == want.shape}
        rep.compare(f"{label}, rounded to 2^{progs.u} == exact", round_to_lattice(got, progs.u), want, others, "lattice words")
        worst = max(worst, max_residual(got, want))
        coef = max(coef, max_coef_sum(progs.cases[ic]["ir"]))
    rep.done()
    assert_residual(progs.p, rep.label, worst, coef)


@pytest.mark.parametrize("threads", MODES, ids=MODE_IDS)
def test_two_programs_two_streams(progs, threads):
    got, _ = _program_schedule(progs, [(0, 0), (1, 1)], threads)
    _check_programs(progs, Report(f"string_contains and pstring_split on two streams, {MODE_IDS[threads]}"),
                    [(progs.cases[0]["label"], 0, got[0]), (progs.cases[1]["label"], 1, got[1])])


def test_one_program_two_streams(progs):
    """one program object (one arena), two inputs"""
    got, _ = _program_schedule(progs, [(1, 1), (1, 2)], False)
    _check_programs(progs, Report("pstring_split, one program on two streams"),
                    [("inputs 1, stream A", 1, got[0]), ("inputs 2, stream B", 2, got[1])])


def test_program_host_run_during_device_run(progs):
    """Program.run (host entry, context stream) of the same program while its program_run_device call is pending on another stream"""
    got, host_out = _program_schedule(progs, [(1, 1)], False, host=(1, 2))
    _check_programs(progs, Report("pstring_split: Program.run while program_run_device is pending"),
                    [("program_run_device, inputs 1", 1, got[0]), ("Program.run, inputs 2", 2, host_out)])
