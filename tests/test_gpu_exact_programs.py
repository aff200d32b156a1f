"""Whole programs word for word on the GPU (run with -m gpu): the level executor (enqueue_levels: linear_kernel, the keyswitch through
in_slot, the fused u16 modulus-switch hand-off, the PBS cut by plan_classic_level with per-launch offsets on lut_idx, out_slot and the
input stride, gather_rows_kernel) against an exact integer executor on the CPU.

Decryption cannot see a row that got the wrong LUT or slot but decrypts to the same message, a coefficient truncated to 32 bits, or an
offset that is wrong only in the third launch of a cut.  Here every word that can reach a keyswitch sits on the coarse lattice 2^u,
u = 63 - log2 N (DESIGN section 4): a lattice BSK on 2^(64 - B_pbs), the program's own accumulators, inputs on 2^u and a test KSK whose body
column is on 2^u.  Then the GPU outputs rounded to 2^u must equal tests/helpers.run_program_exact with orc.pbs_exact_batch on every
word; tests/test_program_exact_premise.py checks the premise on the CPU.  On a mismatch the program is replayed level by level through
Engine.ks_pbs_batch on the exact executor's inputs of each level, which names the first failing level and row and says whether the
kernel or the executor is at fault.
"""
import ctypes as C
import os
import time
from concurrent.futures import ThreadPoolExecutor
from contextlib import contextmanager

import numpy as np
import pytest

from fhe_string_bounty_b200.host import Program
from helpers import (ProgramTrace, coarse_bsk_shift, coarse_headroom_log2, coarse_inputs, coarse_ksk, coarse_shift, engine_params, lattice_bsk,
                     max_coef_sum, max_residual, modulus_switched, round_to_lattice, run_program_exact)

pytestmark = pytest.mark.gpu


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@contextmanager
def _env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


# one program per op family of tfhe_b200_program_build at 2_2 (op, integer arguments, clear operand)
PROGRAMS_2_2 = [
    ("string_eq", (6, 6), None), ("string_ne_packed", (6, 6), None), ("string_lt", (8, 8), None), ("string_le_packed", (6, 6), None),
    ("string_gt", (6,), "abcdez"), ("string_ge", (6, 6), None),
    ("string_contains", (96, 8), None), ("string_contains_packed", (12, 3), None), ("string_starts_with", (12,), "abc"),
    ("string_ends_with", (12, 3), None),
    ("string_find", (24, 3), None), ("string_rfind", (16,), "ab"), ("string_to_lowercase", (8,), None), ("string_to_uppercase", (8,), None),
    ("string_eq_ignore_case", (6, 6), None), ("string_eq_many", (8, 8, 19), None),
    ("radix_add", (8,), None), ("radix_if_then_else", (8,), None), ("radix_full_propagate", (8, 6), None), ("radix_default_lt", (8, 6), None),
    ("radix_scalar_gt", (8, 12345), None),
    ("bool_sum_finish", (3, 1), None), ("signs_finish", (3, 1, 0), None), ("find_combine", (2, 4), None),
    ("pstring_len", (8,), None), ("pstring_trim", (8,), None), ("pstring_find", (8, 2), None), ("pstring_replace", (8, 2, 2), None),
    ("pstring_split", (8, 2), None),
]

# the other kernel families: set -> programs
OTHER_FAMILIES = {
    "multibit_2_2_g3": [("string_lt", (32, 32), None), ("string_le", (32, 32), None), ("string_contains", (12, 3), None)],
    "1_1": [("string_eq", (20, 20), None)],                 # first level 160 >= SM count: pbs_n512; the narrower ones: pbs_generic
    "3_3": [("string_eq", (4, 4), None), ("string_contains", (4, 2), None)],      # pbs_n8192
    "1_3": [("string_eq", (4, 4), None), ("string_lt", (4, 4), None)],            # message modulus 2 on the N = 2048 kernels
    "2_3": [("string_eq", (4, 4), None), ("string_contains", (4, 2), None)],      # pbs_generic, N = 4096
}

SEED_2_2 = 0xF200


def coarse_keys(orc, p, seed, nnz=4):
    """(BSK, KSK) of the coarse lattice, rebuilt from the seed (the sharded reference's worker processes build the same keys)"""
    return lattice_bsk(orc, p, seed, nnz=nnz, shift=coarse_bsk_shift(p)), coarse_ksk(p, seed + 1)


class ExactPrograms:
    """coarse keys of one parameter set, and every program's inputs, exact outputs and level trace"""

    def __init__(self, orc, name, seed, specs, nnz=4):
        self.orc, self.name = orc, name
        self.p = p = orc.params(name)
        self.u = coarse_shift(p)
        self.bsk, self.ksk = coarse_keys(orc, p, seed, nnz)
        self.cases = []
        t0, n_pbs = time.time(), 0
        for i, (op, args, clear) in enumerate(specs):
            P = Program(op, args, clear=clear, params=engine_params(p))
            ir, accs = P.ir(), P.accumulators()
            ins = coarse_inputs(p, P.n_inputs, seed + 100 + i)
            trace = ProgramTrace()
            exact = run_program_exact(orc, ir, accs, p, self.ksk, ins, self.exact_pbs, trace)
            assert not (exact % np.uint64(2**self.u)).any(), f"{op}{args}: an exact output left the 2^{self.u} lattice"
            self.cases.append(dict(label=f"{op}{args}" + (f" clear {clear!r}" if clear else ""), P=P, ir=ir, accs=accs, ins=ins,
                                   exact=exact, trace=trace))
            n_pbs += P.n_pbs
        print(f"[{name}] exact executor: {len(self.cases)} programs, {n_pbs} PBS in {time.time() - t0:.1f} s")

    def exact_pbs(self, small, accs, idx):
        return self.orc.pbs_exact_batch(self.p, self.bsk, small, accs, idx)

    def engine(self, env=None, tuning=None):
        import fhe_string_bounty_b200 as F
        with _env(**(env or {})):
            e = F.Engine(engine_params(self.p))
        for k, v in (tuning or {}).items():      # ks_kernel must be chosen before the KSK is uploaded
            e.set_tuning(k, v)
        e.upload_ksk(self.ksk)
        e.upload_bsk_std(self.bsk)
        return e

    def check(self, eng, variant, device=False):
        """every program on `eng` (and through program_run_device if `device`): outputs rounded to 2^u == the exact executor's, word
        for word; max residual * max sum|coef| below 2^(headroom - 4), as in the CPU premise test"""
        worst, coef = 0, 1
        for c in self.cases:
            runs = [("Program.run", c["P"].run(eng, c["ins"]))]
            if device:
                runs.append(("run_device", _run_device(eng, c["P"], c["ins"])))
            for how, got in runs:
                self._compare(eng, c, got, f"{variant}, {how}")
                worst = max(worst, max_residual(got, c["exact"]))
            coef = max(coef, max_coef_sum(c["ir"]))
        assert_residual(self.p, f"[{self.name}] {variant}: {len(self.cases)} programs, "
                        f"{sum(c['exact'].size for c in self.cases) * (2 if device else 1)} output words", worst, coef)

    def _compare(self, eng, c, got, variant):
        bad = round_to_lattice(got, self.u) != c["exact"]
        if bad.any():
            rows = np.flatnonzero(bad.any(axis=1))
            raise AssertionError(f"[{self.name}] {c['label']} ({variant}): {int(bad.sum())} words in {len(rows)} of {len(got)} output rows "
                                 f"leave the exact executor (first rows {rows[:8].tolist()}); {self._locate(eng, c)}")

    def _locate(self, eng, c):
        """replay each level alone through Engine.keyswitch_batch / ks_pbs_batch on the exact executor's inputs of that level"""
        eng.upload_luts(c["accs"])
        tr, ir = c["trace"], c["ir"]
        for k, lv in enumerate(tr.levels):
            big, idx = tr.big_in[k], tr.lut_idx[k]
            small = eng.keyswitch_batch(big)
            bad_ks = np.flatnonzero((small[:, :-1] != tr.small[k][:, :-1]).any(axis=1)
                                    | (modulus_switched(self.p, small) != modulus_switched(self.p, tr.small[k])).any(axis=1))
            if len(bad_ks):
                return f"keyswitch kernel at fault: level {lv}, row {int(bad_ks[0])} of {len(big)} (pbs job {ir.pbs[int(ir.level_pbs_off[lv]) + int(bad_ks[0])].tolist()})"
            out = eng.ks_pbs_batch(big, idx)
            bad = np.flatnonzero((round_to_lattice(out, self.u) != tr.pbs_out[k]).any(axis=1))
            if len(bad):
                r = int(bad[0])
                return (f"KS-PBS kernel at fault: level {lv} (width {len(big)}), row {r} (in_slot, out_slot, lut = "
                        f"{ir.pbs[int(ir.level_pbs_off[lv]) + r].tolist()})")
        return "every level matches when run alone: the level executor is at fault"


def assert_residual(p, label, worst, coef):
    bound = coarse_headroom_log2(p) - 4
    print(f"{label}, 0 mismatches; max residual 2^{np.log2(max(worst, 1)):.1f} x max sum|coef| {coef} = "
          f"2^{np.log2(max(worst, 1) * coef):.1f} (bound 2^{bound})")
    assert worst * coef < 2**bound, (label, np.log2(max(worst, 1) * coef))


def _run_device(eng, P, ins):
    import torch
    from fhe_string_bounty_b200.multi_gpu import DeviceComm
    comm = DeviceComm(eng, rank=0, world=1)
    with torch.cuda.stream(torch.cuda.Stream()):
        out = comm.to_host(comm.run(P, ins))
    comm.close()
    return out


@pytest.fixture(scope="module")
def progs_2_2(orc):
    return ExactPrograms(orc, "2_2", SEED_2_2, PROGRAMS_2_2)


def test_2_2_tuned_fused(progs_2_2):
    """the default engine: keyswitch on tcgen05 with the fused u16 hand-off, pbs_v4 <4> / <3> and the narrow kernels; Program.run and
    program_run_device"""
    eng = progs_2_2.engine()
    progs_2_2.check(eng, "tuned, fused KS -> PBS", device=True)
    eng.close()


def _plan(batch, sms):
    from fhe_string_bounty_b200._native import load_native
    counts = (C.c_size_t * 3)()
    load_native().tfhe_b200_plan_classic_level(batch, sms, 2 * sms, 1, counts)
    return tuple(int(x) for x in counts)


def _regime(w, sms):
    four, three, tail = _plan(w, sms)
    out = set()
    if not four and not three:
        out.add("v8x2 (<= SMs/2)" if tail <= sms // 2 else "v8 (<= SMs)" if tail <= sms else "v8, 2 per SM (<= 2 SMs)")
    if three:
        out.add("cut with v4<3>")
    if four and tail:
        out.add("v4<4> + tail")
    if four > 4 * sms:
        out.add("two or more waves of four")
    return out


def test_2_2_level_regimes(progs_2_2):
    """the chosen programs drive every cut plan_classic_level makes on this GPU"""
    sms = _sms()
    assert Program("string_contains", (96, 8)).level_widths[0] == (96 - 8 + 1) * 8 * 4 == 2848    # windows x pattern chars x blocks
    assert Program("string_contains", (256, 16)).level_widths[0] == (256 - 16 + 1) * 16 * 4 == 15424
    seen = {}
    for c in progs_2_2.cases:
        for w in c["ir"].level_widths:
            for r in _regime(w, sms):
                seen.setdefault(r, f"{c['label']} level of {w} -> {_plan(w, sms)}")
    for r, where in sorted(seen.items()):
        print(f"regime {r}: {where}")
    want = {"v8x2 (<= SMs/2)", "v8 (<= SMs)", "v8, 2 per SM (<= 2 SMs)", "cut with v4<3>", "v4<4> + tail", "two or more waves of four"}
    assert want <= set(seen), sorted(want - set(seen))


VARIANTS = [
    ("ks_kernel=1 (mma.sync keyswitch, fused)", {}, {"ks_kernel": 1}),
    ("ks_kernel=0 (IMAD keyswitch, unfused hand-off)", {}, {"ks_kernel": 0}),
    ("narrow_kernel=0", {}, {"narrow_kernel": 0}),
    ("narrow_cluster=0", {}, {"narrow_cluster": 0}),
    ("TFHE_B200_PBS_KERNEL=generic", {"TFHE_B200_PBS_KERNEL": "generic"}, {}),
]


@pytest.mark.parametrize("variant", VARIANTS, ids=[v[0].split(" ")[0] for v in VARIANTS])
def test_2_2_variant_settings(progs_2_2, variant):
    label, env, tuning = variant
    eng = progs_2_2.engine(env=env, tuning=tuning)
    progs_2_2.check(eng, label)
    eng.close()


@pytest.mark.parametrize("name", list(OTHER_FAMILIES))
def test_other_kernel_families(orc, name):
    progs = ExactPrograms(orc, name, 0xF300, OTHER_FAMILIES[name])
    if name == "1_1":      # pbs_n512 serves levels of at least SM count ciphertexts
        assert max(progs.cases[0]["ir"].level_widths) >= _sms()
    eng = progs.engine()
    progs.check(eng, "default kernels")
    eng.close()


# ---- sharded operations: DeviceComm.local_group (world ranks on one GPU, exchange kernel) against multi_gpu.sharded_* driven by the
#      exact executor through HostComm in a gloo process group, rank for rank ------------------------------------------------------------

def _sharded_inputs(p):
    """coarse big LWEs: a 12-char haystack and a 3-char pattern, two 8-char strings, and an 8-char string to convert"""
    bpc = 4
    return {k: coarse_inputs(p, bpc * n, 0xF400 + i) for i, (k, n) in enumerate((("hay", 12), ("pat", 3), ("a", 8), ("b", 8), ("s", 8)))}


def _sharded_cases(params, x):
    from fhe_string_bounty_b200 import multi_gpu as MG
    hay, pat, a, b, s = x["hay"], x["pat"], x["a"], x["b"], x["s"]
    cases = [("contains", lambda c: MG.sharded_contains(c, params, hay, pat, 12, 3)),
             ("find", lambda c: MG.sharded_find(c, params, hay, pat, 12, 3)),
             ("eq", lambda c: MG.sharded_eq(c, params, a, b, 8))]
    cases += [(op, lambda c, op=op: MG.sharded_compare(c, params, op, a, b, 8)) for op in ("lt", "le", "gt", "ge")]
    cases += [("to_uppercase", lambda c: MG.sharded_case(c, params, "to_uppercase", s, 8)),
              ("to_lowercase, own share", lambda c: MG.sharded_case(c, params, "to_lowercase", s, 8, gather=False))]
    return cases


def _sharded_worker(rank, world, port, ret):
    """one rank of the exact reference: the same coarse keys from the seed, programs on run_program_exact, collectives over gloo"""
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    sys.path[:0] = [str(root), str(root / "tests")]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), OMP_NUM_THREADS=str(max(1, (os.cpu_count() or 1) // world)))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle import oracle as O
    from fhe_string_bounty_b200.multi_gpu import HostComm
    p = O.params("2_2")
    bsk, ksk = coarse_keys(O, p, SEED_2_2)
    pbs = lambda small, accs, idx: O.pbs_exact_batch(p, bsk, small, accs, idx)
    comm = HostComm(lambda prog, ins: run_program_exact(O, prog.ir(), prog.accumulators(), p, ksk, ins, pbs))
    ret[rank] = [np.atleast_2d(fn(comm)) for _, fn in _sharded_cases(engine_params(p), _sharded_inputs(p))]
    dist.barrier()
    dist.destroy_process_group()


def _free_port():
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


@pytest.mark.parametrize("world", [2, 3])
def test_2_2_sharded_local_group(progs_2_2, world):
    import torch
    import torch.multiprocessing as mp
    from fhe_string_bounty_b200 import multi_gpu as MG
    mgr = mp.get_context("spawn").Manager()       # not a fork of this multi-threaded CUDA process
    ret = mgr.dict()
    t0 = time.time()
    mp.spawn(_sharded_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    exact = [ret[r] for r in range(world)]
    mgr.shutdown()
    print(f"[2_2] sharded, world {world}: exact reference on {world} gloo ranks in {time.time() - t0:.1f} s")
    p, u = progs_2_2.p, progs_2_2.u
    cases = _sharded_cases(engine_params(p), _sharded_inputs(p))
    engines = [progs_2_2.engine() for _ in range(world)]
    comms = MG.DeviceComm.local_group(engines)
    for c in comms:
        c.min_shard_width = 0                        # shard these small trees: the test is about the sharded path
    streams = [torch.cuda.Stream() for _ in comms]

    def all_ranks(fn):
        def one(r):
            with torch.cuda.stream(streams[r]):
                return np.atleast_2d(fn(comms[r]))
        with ThreadPoolExecutor(world) as pool:
            return list(pool.map(one, range(world)))

    got = [[] for _ in range(world)]
    for _, fn in cases:
        for r, out in enumerate(all_ranks(fn)):
            got[r].append(out)
    # the all-reduce adds `world` PBS outputs before bool_sum_finish: that sum carries world * eps like a linear instruction
    coef = max([world] + [max_coef_sum(P.ir()) for c in comms for P in c._programs.values()])
    for c in comms:
        c.close()
    for e in engines:
        e.close()
    for r in range(world):
        worst = 0
        for (label, _), g, want in zip(cases, got[r], exact[r]):
            assert not (want % np.uint64(2**u)).any(), f"sharded {label}: an exact output left the 2^{u} lattice"
            bad = round_to_lattice(g, u) != want
            assert g.shape == want.shape and not bad.any(), \
                f"sharded {label}, world {world}, rank {r}: {int(bad.sum())} words in rows {np.flatnonzero(bad.any(axis=1))[:8].tolist()}"
            worst = max(worst, max_residual(g, want))
        assert_residual(p, f"[2_2] sharded, world {world}, rank {r}: {len(cases)} ops, {sum(w.size for w in exact[r])} output words",
                        worst, coef)
