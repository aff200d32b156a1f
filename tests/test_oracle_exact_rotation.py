"""The exact blind rotation of the oracle (orc_pbs_exact_steps / orc_pbs_exact_batch) and the premise of the word-exact GPU test
(test_gpu_exact_rotation.py, DESIGN section 4): with lattice-valued keys and LUTs, the f64 PBS rounded to 2^s IS the exact integer PBS.

  * classic: the new path equals orc_pbs_exact bit for bit on real (dense) keys;
  * multi-bit: the exact PBS decrypts to the LUT value for every message on real keys, its phase next to the f64 PBS's;
  * every classic and multi-bit parameter set: oracle f64 PBS, rounded to the lattice, equals the exact PBS word for word, residual
    printed and bounded by 2^(s-4) -- with digit-tie LUT words, edge mask words and modulus-switch ties in the inputs;
  * the bisect helper the GPU test uses names the step at which a candidate leaves the exact rotation.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O
from helpers import (assert_on_lattice, first_bad_step, lattice_bsk, lattice_inputs, lattice_luts, lattice_shift, pbs_steps,
                     round_to_lattice)


def test_exact_steps_equals_orc_pbs_exact_classic(orc, toy_keys, keys_2_2):
    """dense real keys: toy set over all 16 messages, and one 2_2 ciphertext whose mask is zero apart from 40 elements (orc_pbs_exact
    costs N^2 per product on a dense key; zero mask elements are skipped by both paths)"""
    p, ck, sk = toy_keys
    acc, _ = sk.generate_lookup_table(lambda x: (3 * x + 1) % 16)
    small = np.stack([sk.keyswitch(ck.encrypt_with_carry(v)) for v in range(16)])
    new = orc.pbs_exact_batch(p, sk.bsk, small, acc[None, :])
    old = np.stack([sk.pbs(x, acc, exact=True) for x in small])
    assert np.array_equal(new, old)
    assert list(ck.decrypt_batch(new)) == [(3 * v + 1) % 16 for v in range(16)]
    one = np.zeros(p.big_dim + 1, dtype=np.uint64)
    orc.lib().orc_pbs_exact_steps(C.byref(p), sk.bsk, small[5], acc, one, C.c_size_t(-1).value)
    assert np.array_equal(one, old[5])

    p, ck, sk = keys_2_2
    acc, _ = sk.generate_lookup_table(lambda x: (5 * x + 2) % 16)
    x = sk.keyswitch(ck.encrypt_with_carry(7))
    keep = np.zeros(p.lwe_dim, dtype=bool)
    keep[np.random.default_rng(3).choice(p.lwe_dim, 38, replace=False)] = True
    keep[[0, p.lwe_dim - 1]] = True
    x[:p.lwe_dim][~keep] = 0
    assert np.array_equal(orc.pbs_exact_batch(p, sk.bsk, x[None, :], acc[None, :])[0], sk.pbs(x, acc, exact=True))


@pytest.mark.parametrize("name", ["multibit_1_1_g2", "multibit_1_1_g3"])
def test_exact_multi_bit_decrypts(orc, name):
    """the exact multi-bit PBS (combined GGSW by exact monomial products, dst = 0; dst += G (x) src) on real keys: every message decrypts
    to the LUT value, and its phase is near the oracle's f64 multi-bit PBS on the same inputs.  With real keys the two differ by more than
    the FFT error: a rounding difference flips level-1 digits (2^(64-B) apart) in the next group, so the bound is a noise-level one,
    a sixteenth of the decoding margin."""
    p = orc.params(name)
    ck = orc.ClientKey(p, 0xB200 + 60)
    sk = orc.ServerKey(ck, 0xB300 + 60)
    space = p.msg_mod * p.carry_mod
    acc, _ = sk.generate_lookup_table(lambda x: (x + 1) % space)
    small = np.stack([sk.keyswitch(ck.encrypt_with_carry(v)) for v in range(space)])
    ex = orc.pbs_exact_batch(p, sk.bsk, small, acc[None, :])
    f64 = np.stack([sk.pbs(x, acc) for x in small])
    assert list(ck.decrypt_batch(ex)) == [(v + 1) % space for v in range(space)]
    assert list(ck.decrypt_batch(f64)) == [(v + 1) % space for v in range(space)]
    d = [abs(((ck.decrypt_raw(a) - ck.decrypt_raw(b)) + 2**63) % 2**64 - 2**63) for a, b in zip(ex, f64)]
    print(f"{name}: |phase(exact) - phase(f64)| max 2^{np.log2(max(max(d), 1)):.1f}")
    assert max(d) < 2**63 // space // 2 // 16


PREMISE_SETS = ["2_2", *O.OTHER_CLASSIC_SETS, "multibit_2_2_g3", *O.OTHER_MULTI_BIT_SETS]


@pytest.mark.parametrize("name", PREMISE_SETS)
def test_lattice_premise(orc, name):
    """sparse lattice key (8 nonzeros per polynomial), tie-crafted LUTs, edge inputs: oracle f64 PBS rounded to 2^s == exact PBS, every
    word of every row; residual <= 2^(s-4).  On a mismatch the failing step is named (bisect over max_steps)."""
    p = orc.params(name)
    s = lattice_shift(p)
    bsk = lattice_bsk(orc, p, seed=11, nnz=8)
    luts = lattice_luts(p, 3, seed=12)
    rows = 8 if p.poly_size <= 8192 else 4
    small = lattice_inputs(p, rows, seed=13)
    idx = (np.arange(rows) % 3).astype(np.uint32)
    fk = orc.FourierKey(p, bsk)
    exact = orc.pbs_exact_batch(p, bsk, small, luts, idx)
    assert not (exact & np.uint64((1 << s) - 1)).any(), "the exact PBS left the lattice"
    got = orc.pbs_f64_batch(p, fk, small, luts, idx)
    assert_on_lattice(got, exact, s, f"oracle f64 {name} (N={p.poly_size} k={p.glwe_dim} l={p.pbs_level} B={p.pbs_base_log})",
                      run_rows=lambda k, r: orc.pbs_f64_batch(p, fk, small[r], luts, idx[r], max_steps=k),
                      ref_rows=lambda k, r: orc.pbs_exact_batch(p, bsk, small[r], luts, idx[r], max_steps=k),
                      n_steps=pbs_steps(p))


@pytest.mark.parametrize("name", ["1_1", "2_2"])
def test_lattice_premise_dense_key(orc, name):
    """the premise on a dense lattice key (every coefficient in [-127, 127] * 2^s): the FFT error grows with the key's weight and
    still stays far below the half lattice"""
    p = orc.params(name)
    s = lattice_shift(p)
    bsk = lattice_bsk(orc, p, seed=21, nnz=None)
    luts = lattice_luts(p, 2, seed=22)
    small = lattice_inputs(p, 2, seed=23)
    small[:, :p.lwe_dim][:, 64:] = 0     # the dense exact product costs N^2 per polynomial: 64 steps (zero mask elements are skipped)
    idx = np.array([0, 1], dtype=np.uint32)
    exact = orc.pbs_exact_batch(p, bsk, small, luts, idx)
    got = orc.pbs_f64_batch(p, orc.FourierKey(p, bsk), small, luts, idx)
    assert_on_lattice(got, exact, s, f"oracle f64 {name}, dense lattice key")


def test_bisect_names_the_perturbed_step(orc):
    """a candidate that uses the wrong GGSW at one step (index j0 + 1 in place of j0) leaves the exact rotation at step j0 + 1; the
    helper shared with the GPU test must report that step, the row and a nonzero word count"""
    for name, j0 in (("1_1", 37), ("multibit_1_1_g3", 200)):
        p = orc.params(name)
        s = lattice_shift(p)
        bsk = lattice_bsk(orc, p, seed=31)
        step = ((1 << p.grouping_factor) if p.grouping_factor else 1) * p.pbs_level * (p.glwe_dim + 1)**2 * p.poly_size   # words per step
        bad = bsk.copy()
        bad[j0 * step:(j0 + 1) * step] = bsk[(j0 + 1) * step:(j0 + 2) * step]
        luts = lattice_luts(p, 1, seed=32)
        small = lattice_inputs(p, 4, seed=33)[3:]
        small[0, j0 * max(p.grouping_factor, 1)] = 0x5A5A5A5A5A5A5A5A     # a classic PBS skips a zero mask element
        run = lambda k: orc.pbs_exact_batch(p, bad, small, luts, max_steps=k)[0]
        ref = lambda k: orc.pbs_exact_batch(p, bsk, small, luts, max_steps=k)[0]
        assert (round_to_lattice(run(None), s) != ref(None)).any()
        k, words = first_bad_step(run, ref, pbs_steps(p), s)
        assert k == j0 + 1 and words > 0, (name, k, words)
        with pytest.raises(AssertionError, match=f"row 0 first differs after step {j0 + 1} of {pbs_steps(p)}"):
            assert_on_lattice(run(None)[None, :], ref(None)[None, :], s, name,
                              run_rows=lambda k, r: orc.pbs_exact_batch(p, bad, small[r], luts, max_steps=k),
                              ref_rows=lambda k, r: orc.pbs_exact_batch(p, bsk, small[r], luts, max_steps=k), n_steps=pbs_steps(p))
