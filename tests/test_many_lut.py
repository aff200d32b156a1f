"""Many-LUT accumulators (tfhe-rs generate_many_lookup_table) without a GPU: many_lut_accumulator is byte-equal to the oracle's
generate_lookup_table of the stacked table (box f * chunk + x holds f_f(x), zero from F * chunk on), the refusals of F out of range, and
the extraction-at-t reference of the GPU tests against a direct restatement."""
import numpy as np
import pytest

from many_lut_ref import extract_mask_at, mask_from_row0


def _fns(F, msg_mod, seed):
    rng = np.random.default_rng(seed)
    tables = rng.integers(0, msg_mod, size=(F, 256))
    return [(lambda x, t=t: int(t[x])) for t in tables]


def _stacked(fns, total):
    F = len(fns)
    chunk = total // F
    return lambda i: fns[i // chunk](i % chunk) if i < F * chunk else 0


@pytest.mark.parametrize("name,F", [("2_2", 2), ("2_2", 3), ("2_2", 4), ("1_1", 4), ("3_3", 64), ("3_3", 5), ("2_3", 32), ("4_4", 256)])
def test_accumulator_matches_the_stacked_table(orc, name, F):
    import ctypes as C
    import fhe_string_bounty_b200 as FB
    from helpers import engine_params
    p = orc.params(name)
    total = p.msg_mod * p.carry_mod
    fns = _fns(F, p.msg_mod, 0x3A00 + F)
    got = FB.many_lut_accumulator(engine_params(p), fns)
    table = np.array([_stacked(fns, total)(i) for i in range(total)], dtype=np.uint64)
    want = np.zeros(p.lut_len, dtype=np.uint64)
    orc.lib().orc_fill_accumulator(C.byref(p), table, want)
    assert got.dtype == np.uint64 and got.shape == (p.lut_len,)
    assert np.array_equal(got, want)
    # restated from the definition: box b of the body (before the half-box rotation) holds table[b] * delta
    N, box = p.poly_size, p.poly_size // total
    body = np.roll(got[p.glwe_dim * N:], box // 2)
    body[:box // 2] = np.uint64(0) - body[:box // 2]
    delta = (1 << 63) // total
    assert all(int(body[b * box]) == (int(table[b]) * delta) % 2**64 for b in range(total))
    assert not got[:p.glwe_dim * N].any()


@pytest.mark.parametrize("F", [0, 1, 17])
def test_function_count_out_of_range_is_refused(orc, F):
    import fhe_string_bounty_b200 as FB
    from helpers import engine_params
    p = orc.params("2_2")         # total 16
    with pytest.raises(ValueError, match="functions"):
        FB.many_lut_accumulator(engine_params(p), [lambda x: 0] * F)


@pytest.mark.parametrize("t", [0, 1, 511, 1024, 2047])
def test_extraction_reference(orc, t):
    """extract_mask_at(mask_from_row0(row0), t) == the definition, word by word, on a random two-mask GLWE"""
    p = orc.params("1_2")          # k = 2, N = 1024
    N, k = p.poly_size, p.glwe_dim
    t = t % N
    rng = np.random.default_rng(t)
    A = rng.integers(0, 2**64, size=(k, N), dtype=np.uint64)
    row0 = extract_mask_at(A, 0)
    assert np.array_equal(mask_from_row0(p, row0), A)
    got = extract_mask_at(A, t)
    for r in range(k):
        for q in range(N):
            want = A[r, t - q] if q <= t else (0 - int(A[r, N + t - q])) % 2**64
            assert int(got[r * N + q]) == int(want)


@pytest.mark.parametrize("name,nnz", [("2_2", 8), ("multibit_2_2_g3", 4), ("3_3", 8), ("1_1", 8)])
def test_exact_glwe_reference_matches_the_oracle(orc, name, nnz):
    """the numpy exact blind rotation (classic, multi-bit, two levels, k = 3) extracted at monomial 0 equals orc_pbs_exact_batch word for
    word, after the whole rotation and stopped after a few steps (the bisection of the GPU tests uses both)"""
    from helpers import lattice_bsk, lattice_inputs, lattice_luts
    from many_lut_ref import exact_glwe_batch, extract_at
    p = orc.params(name)
    bsk = lattice_bsk(orc, p, 0x3B00, nnz=nnz)
    luts = lattice_luts(p, 3, 0x3B01)
    small = lattice_inputs(p, 4, 0x3B02)
    idx = (np.arange(4) % 3).astype(np.uint32)
    for steps in (None, 3):
        got = extract_at(exact_glwe_batch(p, bsk, small, luts, idx, max_steps=steps), 0)
        assert np.array_equal(got, orc.pbs_exact_batch(p, bsk, small, luts, idx, max_steps=steps)), (name, steps)
