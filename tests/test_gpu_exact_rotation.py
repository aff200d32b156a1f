"""Word-exact parity of the WHOLE blind rotation for every PBS kernel instance (run with -m gpu), on lattice-valued test keys.

With real keys two correct implementations give different full-PBS words (DESIGN section 4), so the other GPU tests compare one step
word by word and the full PBS only after decryption.  Here the BSK is small multiples of 2^s (s = 64 - pbs_base_log * pbs_level, 8
nonzeros per polynomial) and the LUTs are multiples of 2^s with digit-tie words, so every accumulator coefficient stays on the lattice and
the kernel's output rounded to 2^s must equal the oracle's exact integer PBS (orc_pbs_exact_batch) on every word of every row after all n
steps: the TMA key rings and their wrap-around, the prefetch, the cluster spectrum swap, multi-bit combines of every group, ragged tails.
Per kernel instance: (a) rows compared word for word, 0 mismatches -- a mismatch is bisected over n_iters to the first failing step;
(b) max residual |out - exact| (the kernel's FFT error) <= 2^(s-4), printed.  The inputs hold edge mask words (0, 1, 2^64 - 1, 2^63)
and modulus-switch ties.  Instances are pinned by batch size, set_tuning and environment variables, as in test_gpu_wide_kernels.py.

Also: the fused KS -> PBS path (real KSK, and a crafted KSK whose outputs sit exactly on modulus-switch ties, so the u16 epilogue's
rounding meets orc_modulus_switch), PBS -> KS == keyswitch_batch(pbs_batch), and real keys at later key indices (one CMUX with GGSW j,
against the exact external product, DESIGN bound 2^44).
"""
import ctypes as C
import os
from contextlib import contextmanager

import numpy as np
import pytest

from helpers import (assert_on_lattice, engine_params, exact_unique, lattice_bsk, lattice_inputs, lattice_luts, lattice_shift,
                     max_residual, modulus_switch_ties, pbs_steps)

pytestmark = pytest.mark.gpu


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@contextmanager
def _env(**kv):
    """environment variables read at Engine creation (TFHE_B200_*) or at launch"""
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


def _engine(p, bsk, luts, ksk=None, env=None, tuning=None):
    import fhe_string_bounty_b200 as F
    with _env(**(env or {})):
        e = F.Engine(engine_params(p))
    if ksk is not None:
        e.upload_ksk(ksk)
    e.upload_bsk_std(bsk)
    e.upload_luts(luts)
    for k, v in (tuning or {}).items():
        e.set_tuning(k, v)
    return e


class LatticeCase:
    """lattice BSK + LUTs + an input pool of one parameter set; the exact reference is computed once for the pool's distinct rows"""

    def __init__(self, orc, name, seed, pool, nnz=8, n_luts=3):
        self.orc, self.name = orc, name
        self.p = p = orc.params(name)
        self.s = lattice_shift(p)
        self.bsk = lattice_bsk(orc, p, seed, nnz=nnz)
        self.luts = lattice_luts(p, n_luts, seed + 1)
        self.small = lattice_inputs(p, pool, seed + 2)
        self.idx = ((np.arange(pool) * 7 + np.arange(pool) // 64) % n_luts).astype(np.uint32)
        self.exact = exact_unique(orc, p, self.bsk, self.small, self.luts, self.idx)

    def check(self, eng, batch, label, start=0):
        """pbs_batch over `batch` rows of the pool from `start`, (a) and (b) on every row; returns the max residual"""
        p, s = self.p, self.s
        small, idx, exact = self.small[start:start + batch], self.idx[start:start + batch], self.exact[start:start + batch]
        got = eng.pbs_batch(small, idx)
        return assert_on_lattice(
            got, exact, s, f"{label} [{self.name}, batch {batch}]",
            run_rows=lambda k, r: eng.pbs_batch(small, idx, n_iters=k)[r],
            ref_rows=lambda k, r: self.orc.pbs_exact_batch(p, self.bsk, small[r], self.luts, idx[r], max_steps=k),
            n_steps=pbs_steps(p))


@pytest.fixture(scope="module")
def case_2_2(orc):
    sms = _sms()
    return LatticeCase(orc, "2_2", 0xE200, pool=max(5 * sms, 4 * sms + 200))


@pytest.fixture(scope="module")
def case_mb(orc):
    return LatticeCase(orc, "multibit_2_2_g3", 0xE300, pool=3 * _sms() + 2, nnz=4)


def _classic_configs(sms):
    """(label, batch, env, tuning): every classic N = 2048 instance"""
    return [
        ("pbs_classic_kernel_v4<4> + v8 tail", 4 * sms + 3, {}, {}),
        ("pbs_classic_kernel_v4<3>", 3 * sms - 1, {}, {}),
        ("planned cut: two waves of <3> in one launch", 4 * sms + 200, {}, {}),
        ("planned cut: <3> wave + v8 tail", 5 * sms, {}, {}),
        ("pbs_classic_kernel_v4<2>", 2 * sms - 1, {}, {"narrow_kernel": 0}),
        ("pbs_classic_kernel_v4<1>", sms - 1, {}, {"narrow_kernel": 0}),
        ("pbs_classic_kernel_v8 (one SM)", 37, {}, {"narrow_cluster": 0}),
        ("pbs_classic_kernel_v8 (one SM, 2 per SM)", 2 * sms - 3, {}, {"narrow_cluster": 0}),
        ("pbs_classic_kernel_v8x2 (two-SM cluster)", 37, {}, {}),
        ("batch of one", 1, {}, {}),
        ("pbs_generic", 37, {"TFHE_B200_PBS_KERNEL": "generic"}, {}),
    ]


def _start(batch):
    """a batch of one takes pool row 3 (rows 0 ... 2 are the all-zero, all-tie and fixed-edge masks, covered by the wider batches)"""
    return 3 if batch == 1 else 0


def test_classic_2_2_every_instance(case_2_2):
    sms = _sms()
    for label, batch, env, tuning in _classic_configs(sms):
        eng = _engine(case_2_2.p, case_2_2.bsk, case_2_2.luts, env=env, tuning=tuning)
        case_2_2.check(eng, batch, label, start=_start(batch))
        eng.close()


def test_classic_2_2_dense_key_probe_rows(orc, case_2_2):
    """a dense lattice key (every coefficient in [-127, 127] * 2^s) on pbs_classic_kernel_v4<4>: the exact reference costs N^2 per product,
    so only probe rows (first and last CTA, a spread in between) are compared"""
    p, s = case_2_2.p, case_2_2.s
    sms = _sms()
    batch = 4 * sms
    bsk = lattice_bsk(orc, p, 0xE250, nnz=None)
    small, idx, luts = case_2_2.small[:batch], case_2_2.idx[:batch], case_2_2.luts
    small = small.copy()
    small[:, 200:p.lwe_dim] = 0      # 200 nonzero mask elements: a dense exact product costs N^2 per polynomial
    rows = sorted({0, 1, 2, 3, batch // 2, batch // 2 + 1, batch - 4, batch - 3, batch - 2, batch - 1})
    eng = _engine(p, bsk, luts)
    got = eng.pbs_batch(small, idx)
    eng.close()
    exact = orc.pbs_exact_batch(p, bsk, small[rows], luts, idx[rows])
    assert_on_lattice(got[rows], exact, s, f"pbs_classic_kernel_v4<4>, dense lattice key [{len(rows)} probe rows of {batch}]")


def test_multibit_2_2_g3_every_instance(case_mb):
    sms = _sms()
    configs = [
        ("pbs_multibit_kernel_v4<3> + v8 tail", 3 * sms + 2, {}, {}),
        ("pbs_multibit_kernel_v4<2>", 2 * sms - 1, {}, {"narrow_kernel": 0}),
        ("pbs_multibit_kernel_v4<1>", sms - 1, {}, {"narrow_kernel": 0}),
        ("pbs_multibit_kernel_v8 (one SM)", 37, {}, {"narrow_cluster": 0}),
        ("pbs_multibit_kernel_v8x2 (two-SM cluster)", 37, {}, {}),
        ("batch of one", 1, {}, {}),
    ]
    for label, batch, env, tuning in configs:
        eng = _engine(case_mb.p, case_mb.bsk, case_mb.luts, env=env, tuning=tuning)
        case_mb.check(eng, batch, label, start=_start(batch))
        eng.close()


def test_tuned_n512_instances(orc):
    """PARAM_MESSAGE_1_CARRY_1 on pbs_n512.cu: the 1-, 4- and 8-ciphertext instances (tuned512_min = 1)"""
    sms = _sms()
    case = LatticeCase(orc, "1_1", 0xE400, pool=8 * sms + 5)
    eng = _engine(case.p, case.bsk, case.luts, tuning={"tuned512_min": 1})
    for batch, cts in ((3, 1), (sms + 5, 4), (8 * sms + 5, 8)):
        case.check(eng, batch, f"pbs_n512_kernel<{cts}>")
    eng.close()


def test_tuned_n8192(orc):
    """PARAM_MESSAGE_3_CARRY_3 on pbs_n8192.cu (one ciphertext per two-SM cluster), a batch wider than the clusters that fit"""
    sms = _sms()
    case = LatticeCase(orc, "3_3", 0xE500, pool=sms // 2 + 7)
    eng = _engine(case.p, case.bsk, case.luts, tuning={"tuned8192": 1})
    for batch in (3, sms // 2 + 7):
        case.check(eng, batch, "pbs_n8192")
    eng.close()


@pytest.mark.parametrize("name", ["1_0", "2_0", "1_2", "2_3", "1_4", "4_3", "4_4",
                                  "multibit_1_1_g2", "multibit_2_2_g2", "multibit_3_3_g2", "multibit_1_1_g3", "multibit_3_3_g3"])
def test_generic_kernel_shapes(orc, name):
    """pbs_generic.cu on the other shapes (4_3: launch_big<14>, 4_4: launch_big<15>) and the multi-bit sets of grouping factor 2 and 3"""
    p = orc.params(name)
    rows = 24 if p.poly_size <= 4096 else 12 if p.poly_size <= 8192 else 4
    case = LatticeCase(orc, name, 0xE600, pool=rows, nnz=8 if not p.grouping_factor else 4)
    eng = _engine(p, case.bsk, case.luts)
    case.check(eng, rows, "pbs_generic")
    eng.close()


def test_fused_ks_pbs_real_ksk(orc, keys_2_2, case_2_2):
    """ks_pbs_batch (keyswitch epilogue hands the u16 modulus switch to pbs_v4 / pbs_v8) with the real 2_2 KSK and the lattice BSK ==
    oracle keyswitch followed by the exact rotation, every row"""
    p, ck, sk = keys_2_2
    sms = _sms()
    batch = 4 * sms + 3
    rng = np.random.default_rng(0xE700)
    cts = ck.encrypt_batch(rng.integers(0, 16, size=batch))
    small = np.stack([sk.keyswitch(c) for c in cts])
    idx = (np.arange(batch) % len(case_2_2.luts)).astype(np.uint32)
    eng = _engine(p, case_2_2.bsk, case_2_2.luts, ksk=sk.ksk)
    got = eng.ks_pbs_batch(cts, idx)
    assert np.array_equal(eng.keyswitch_batch(cts), small)
    eng.close()
    exact = exact_unique(orc, p, case_2_2.bsk, small, case_2_2.luts, idx)
    assert_on_lattice(got, exact, case_2_2.s, f"fused KS -> pbs_classic_kernel_v4<4> + v8 tail, real KSK [batch {batch}]")


def test_fused_ks_pbs_on_modulus_switch_ties(orc, case_2_2):
    """a crafted KSK with one nonzero row (i0, level index j0) and inputs whose only nonzero decomposition digit selects it with +-1: the
    keyswitch output is -+row exactly, a row of modulus-switch ties (and 0, 2^63, 2^64 - 1), so the fused u16 epilogue must round every
    tie as orc_modulus_switch does"""
    p, s = case_2_2.p, case_2_2.s
    L, B, n = p.ks_level, p.ks_base_log, p.lwe_dim
    rng = np.random.default_rng(0xE800)
    i0, j0 = 1000, 2                                   # level index j0 holds level L - j0 (levels stored L .. 1)
    ksk = np.zeros((p.big_dim, L, n + 1), dtype=np.uint64)
    row = modulus_switch_ties(p, rng, n + 1)
    row[:4] = np.array([0, 2**63, 2**64 - 1, 1], dtype=np.uint64)
    ksk[i0, j0] = row
    sms = _sms()
    uniq = np.zeros((8, p.big_dim + 1), dtype=np.uint64)
    one = 1 << (64 - B * (L - j0))                     # digit +1 at level L - j0
    for u in range(8):
        uniq[u, i0] = one if u % 2 == 0 else 2**64 - one
        uniq[u, p.big_dim] = rng.integers(0, 2**64, dtype=np.uint64) if u < 6 else modulus_switch_ties(p, rng, 1)[0]
    ks = np.zeros((8, n + 1), dtype=np.uint64)
    for u in range(8):
        orc.lib().orc_keyswitch(C.byref(p), ksk.ravel(), uniq[u], ks[u])
        want = (np.uint64(0) - row) if u % 2 == 0 else row.copy()
        assert np.array_equal(ks[u][:n], want[:n]), "the crafted input must select the row with digit +-1"
    for batch in (4 * sms + 3, 37):                    # wide v4<4> + v8 tail, and a narrow level on the v8 cluster instance
        cts = uniq[np.arange(batch) % 8]
        small = ks[np.arange(batch) % 8]
        idx = (np.arange(batch) % len(case_2_2.luts)).astype(np.uint32)
        eng = _engine(p, case_2_2.bsk, case_2_2.luts, ksk=ksk.ravel())
        got = eng.ks_pbs_batch(cts, idx)
        assert np.array_equal(eng.keyswitch_batch(cts), small)
        eng.close()
        exact = exact_unique(orc, p, case_2_2.bsk, small, case_2_2.luts, idx)
        assert_on_lattice(got, exact, s, f"fused KS -> PBS, keyswitch outputs on modulus-switch ties [batch {batch}]")


def test_pbs_then_ks_order(keys_2_2, case_2_2):
    """pbs_ks_batch(x) == keyswitch_batch(pbs_batch(x)) word for word (the exact PBS -> KS comparison is not decidable: lattice words can
    sit on keyswitch rounding ties)"""
    p, ck, sk = keys_2_2
    sms = _sms()
    eng = _engine(p, case_2_2.bsk, case_2_2.luts, ksk=sk.ksk)
    for batch in (4 * sms + 3, 37):
        small, idx = case_2_2.small[:batch], case_2_2.idx[:batch]
        assert np.array_equal(eng.pbs_ks_batch(small, idx), eng.keyswitch_batch(eng.pbs_batch(small, idx))), batch
    eng.close()


def test_real_key_late_indices(orc, keys_2_2):
    """real 2_2 keys, small LWEs whose mask is zero except at one index j (j = 0, 1, around the ring sizes 2, 4, 5, 7, 9, 11 of the
    instances, n-2, n-1): every other step leaves the accumulator exactly unchanged, so the full PBS is one CMUX with GGSW j.  Against
    the exact PBS: max |delta| <= 2^44 (DESIGN section 4), printed next to the oracle f64's own distance to the exact result."""
    p, ck, sk = keys_2_2
    n = p.lwe_dim
    js = [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, n - 2, n - 1]
    luts = np.stack([sk.generate_lookup_table(f)[0] for f in (lambda x: x, lambda x: (3 * x + 1) % 16)])
    rng = np.random.default_rng(0xE900)
    uniq = np.zeros((2 * len(js), n + 1), dtype=np.uint64)
    for u in range(len(uniq)):
        uniq[u, js[u % len(js)]] = rng.integers(1, 2**64, dtype=np.uint64)
        uniq[u, n] = rng.integers(0, 2**64, dtype=np.uint64)
    uidx = (np.arange(len(uniq)) // len(js)).astype(np.uint32)
    exact = orc.pbs_exact_batch(p, sk.bsk, uniq, luts, uidx)
    f64 = np.stack([sk.pbs(x, luts[i]) for x, i in zip(uniq, uidx)])
    d_orc = max_residual(f64, exact)
    sms = _sms()
    for label, batch, env, tuning in _classic_configs(sms):
        eng = _engine(p, sk.bsk, luts, env=env, tuning=tuning)
        sel = np.arange(batch) % len(uniq)
        got = eng.pbs_batch(uniq[sel], uidx[sel])
        eng.close()
        d = max_residual(got, exact[sel])
        print(f"{label} [real 2_2 key, batch {batch}]: one CMUX at j in {js}: max |gpu - exact| 2^{np.log2(max(d, 1)):.1f}, "
              f"oracle f64 - exact 2^{np.log2(max(d_orc, 1)):.1f} (bound 2^44)")
        assert d <= 2**44, (label, np.log2(d))
