"""CPU premise of tests/test_gpu_exact_programs.py (no GPU): on the coarse lattice 2^u, u = 63 - log2 N (DESIGN section 4), a whole
program run with a floating-point PBS, rounded to 2^u, equals the exact integer executor on every word.

(a) The replay logic of helpers.run_program_exact, with real toy keys and the oracle's f64 PBS, is oracle/radix.run_program word for
word.  (b) For every parameter set and op family the GPU test runs, at reduced sizes: run_program_exact with orc.pbs_f64_batch (a
FourierKey of the coarse BSK) standing in for the GPU, against the same executor with orc.pbs_exact_batch.  Per level the small LWEs
agree on every mask word and every modulus-switched value, the rounded PBS outputs are exact, and so are the rounded program outputs.
The max f64 residual and the program's largest sum |coef| of one linear instruction are printed, and residual * sum|coef| must stay
16x below the headroom 2^(min(u, 64 - B_ks * l_ks) - 1).
"""
import numpy as np
import pytest

from fhe_string_bounty_b200.host import Program
from helpers import (ProgramTrace, coarse_bsk_shift, coarse_headroom_log2, coarse_inputs, coarse_ksk, coarse_shift, engine_params, lattice_bsk,
                     max_coef_sum, max_residual, modulus_switched, round_to_lattice, run_program_exact)


def test_coarse_lattice_conditions_every_set():
    """u >= 64 - B_pbs * l_pbs, u >= 64 - B_ks * l_ks and delta >= 2^u for all 36 classic and 6 multi-bit sets (coarse_shift asserts them)"""
    from fhe_string_bounty_b200._native import _CLASSIC_SETS, _MULTI_BIT_SETS, Params, classic_params, multi_bit_params
    sets = [classic_params(n) for n in _CLASSIC_SETS] + [multi_bit_params(n) for n in _MULTI_BIT_SETS]
    u = {n: coarse_shift(Params(**kw)) for n, kw in zip(list(_CLASSIC_SETS) + list(_MULTI_BIT_SETS), sets)}
    assert len(u) == 42 and (u["2_2"], u["3_3"], u["4_4"]) == (52, 50, 48)


def test_replay_matches_oracle_run_program(orc, toy_keys):
    from oracle import radix as R
    p, ck, sk = toy_keys
    fourier = orc.FourierKey(p, sk.bsk)
    f64 = lambda small, accs, idx: orc.pbs_f64_batch(p, fourier, small, accs, idx)
    a, b = b"hello", b"help!"
    cases = [("string_lt", (5, 5), None, np.concatenate([R.encrypt_string(ck, a), R.encrypt_string(ck, b)])),
             ("string_find", (5, 2), None, np.concatenate([R.encrypt_string(ck, a), R.encrypt_string(ck, b"lo")])),
             ("string_contains", (5,), "el", R.encrypt_string(ck, a)),
             ("radix_add", (3,), None, np.stack(R.encrypt_radix(ck, 45, 3) + R.encrypt_radix(ck, 27, 3))),
             ("pstring_trim", (4,), None, R.encrypt_string(ck, b" a\0\0"))]
    for op, args, clear, ins in cases:
        P = Program(op, args, clear=clear, params=engine_params(p))
        ir = P.ir()
        want = R.run_program(ir, sk, ins)
        got = run_program_exact(orc, ir, P.accumulators(), p, sk.ksk, ins, f64)
        assert np.array_equal(got, want), op


# every program the GPU test runs, at reduced sizes: (set, [(op, args, clear)])
PREMISE = {
    "2_2": [("string_eq", (4, 4), None), ("string_ne_packed", (3, 3), None), ("string_lt", (4, 4), None), ("string_gt", (4,), "abcz"),
            ("string_contains_packed", (6, 2), None), ("string_starts_with", (6,), "ab"), ("string_ends_with", (6, 2), None),
            ("string_find", (8, 2), None), ("string_rfind", (6,), "ab"), ("string_to_uppercase", (4,), None),
            ("string_eq_ignore_case", (3, 3), None), ("string_eq_many", (2, 2, 3), None),
            ("radix_add", (4,), None), ("radix_if_then_else", (4,), None), ("radix_full_propagate", (4, 6), None),
            ("radix_default_lt", (4, 6), None), ("radix_scalar_gt", (4, 77), None),
            ("bool_sum_finish", (3, 1), None), ("signs_finish", (3, 1, 0), None), ("find_combine", (2, 4), None),
            ("pstring_len", (4,), None), ("pstring_trim", (4,), None), ("pstring_find", (4, 2), None),
            ("string_le_packed", (3, 3), None), ("string_ge", (3, 3), None), ("string_contains", (6, 2), None),
            ("string_to_lowercase", (4,), None), ("pstring_replace", (4, 2, 2), None), ("pstring_split", (4, 2), None),
            # the rank shares of the sharded operations (their finishing programs are bool_sum_finish, signs_finish, find_combine)
            ("string_contains_windows", (6, 2, 0, 3), None), ("string_find_windows", (8, 2, 2, 5), None), ("string_cmp_sign", (4, 4), None)],
    "multibit_2_2_g3": [("string_lt", (8, 8), None), ("string_le", (8, 8), None), ("string_contains", (6, 2), None)],
    "1_1": [("string_eq", (4, 4), None)],
    "3_3": [("string_eq", (3, 3), None), ("string_contains", (4, 2), None)],
    "1_3": [("string_lt", (4, 4), None), ("string_eq", (4, 4), None)],
    "2_3": [("string_contains", (4, 2), None), ("string_eq", (4, 4), None)],
}


@pytest.mark.parametrize("name", list(PREMISE))
def test_f64_executor_rounds_to_exact(orc, name):
    p = orc.params(name)
    u = coarse_shift(p)
    head = coarse_headroom_log2(p)
    bsk, bsk_other = (lattice_bsk(orc, p, seed, nnz=4, shift=coarse_bsk_shift(p)) for seed in (0xF100, 0xF102))
    ksk = coarse_ksk(p, 0xF101)
    fourier = orc.FourierKey(p, bsk)
    exact_pbs = lambda small, accs, idx: orc.pbs_exact_batch(p, bsk, small, accs, idx)
    f64_pbs = lambda small, accs, idx: orc.pbs_f64_batch(p, fourier, small, accs, idx)
    worst_res, worst_coef = 0, 1
    for i, (op, args, clear) in enumerate(PREMISE[name]):
        P = Program(op, args, clear=clear, params=engine_params(p))
        ir, accs = P.ir(), P.accumulators()
        assert P.n_pbs > 0, op
        ins = coarse_inputs(p, P.n_inputs, 0xF110 + i)
        te, tf = ProgramTrace(), ProgramTrace()
        exact = run_program_exact(orc, ir, accs, p, ksk, ins, exact_pbs, te)
        got = run_program_exact(orc, ir, accs, p, ksk, ins, f64_pbs, tf)
        assert not (exact % np.uint64(2**u)).any(), f"{op}: exact output off the 2^{u} lattice"
        res = 0
        for k, lv in enumerate(te.levels):
            se, sf = te.small[k], tf.small[k]
            assert np.array_equal(sf[:, :-1], se[:, :-1]), f"{op} level {lv}: small mask words differ"
            assert np.array_equal(modulus_switched(p, sf), modulus_switched(p, se)), f"{op} level {lv}: modulus-switched values differ"
            assert np.array_equal(round_to_lattice(tf.pbs_out[k], u), te.pbs_out[k]), f"{op} level {lv}: rounded PBS outputs differ"
            res = max(res, max_residual(tf.pbs_out[k], te.pbs_out[k]))
        assert np.array_equal(round_to_lattice(got, u), exact), f"{op}: rounded outputs differ"
        if i == 0:      # the outputs depend on the BSK: the external products do not vanish modulo 2^64 on the lattice
            other = run_program_exact(orc, ir, accs, p, ksk, ins, lambda s, a, j: orc.pbs_exact_batch(p, bsk_other, s, a, j))
            assert not np.array_equal(other, exact), f"{op}: the outputs do not depend on the BSK"
        coef = max_coef_sum(ir)
        print(f"[{name}] {op}{args}: {P.n_pbs} PBS, {len(ir.level_widths)} levels, f64 residual 2^{np.log2(max(res, 1)):.1f}, "
              f"max sum|coef| {coef}")
        worst_res, worst_coef = max(worst_res, res), max(worst_coef, coef)
    margin = np.log2(max(worst_res, 1) * worst_coef)
    print(f"[{name}] u = {u}, headroom 2^{head}: max residual 2^{np.log2(max(worst_res, 1)):.1f} x max sum|coef| {worst_coef} "
          f"= 2^{margin:.1f} (bound 2^{head - 4})")
    assert worst_res * worst_coef < 2**(head - 4), (name, margin)
