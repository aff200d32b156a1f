"""Word-exact parity over the accepted parameter range, not only at the named sets (run with -m gpu).

The kernel is chosen from (N, k, l, g) alone, so any accepted LWE dimension and base log of a tuned shape runs the tuned kernel.  Here:

  * keyswitch: every accepted (base_log, level) with level <= 7 on ks_kernel 2 (tcgen05), 1 (mma.sync) and 0 (IMAD), and levels 8 ... 13
    on the IMAD kernel (the only one above 7), at output widths n + 1 around the 128-column tiles, on kN = 2048 and 32768, word for word
    against orc_keyswitch; the all-0xFF key at (7, 4) and (6, 5) on kN = 32768, where the tensor-core plane sums pass 2^31; the fused u16
    modulus-switch epilogue (ks_pbs_batch) at odd and even row strides;
  * blind rotation: every point of param_range.py on every kernel instance its shape has (pinned by batch size and tuning), word for word
    against the exact rotation on lattice-valued keys (DESIGN section 4), a mismatch bisected to its first failing step;
  * contexts: a context created later with fewer keyswitch levels leaves an earlier context's IMAD keyswitch working, and level counts
    the IMAD kernel cannot stage in shared memory are refused with a message that names the limit.

Wide batches repeat a pool of 37 distinct rows (row i = pool[i mod 37]; 37 is prime to the 2, 3, 4 and 8 ciphertexts per CTA, so every
CTA holds distinct rows and a swap between its ciphertexts shows); the exact reference is computed once per distinct row."""
import os
from contextlib import contextmanager

import numpy as np
import pytest

from helpers import (assert_on_lattice, engine_params, exact_unique, keyswitch_rows, lattice_bsk, lattice_inputs, lattice_luts,
                     lattice_shift, pbs_steps)
from param_range import CLASSIC, GENERIC, MULTIBIT, N512, N8192, Point
from test_gpu_all_param_sets import BATCHES, ks_inputs, max_digit_word, probe_rows

pytestmark = pytest.mark.gpu

POOL = 37


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


def _params(orc, N, k, n, ks_base_log, ks_level, pbs_base_log=15, pbs_level=2):
    p = orc.Params()
    p.lwe_dim, p.glwe_dim, p.poly_size, p.pbs_base_log, p.pbs_level = n, k, N, pbs_base_log, pbs_level
    p.ks_base_log, p.ks_level, p.grouping_factor, p.msg_mod, p.carry_mod = ks_base_log, ks_level, 0, 4, 4
    return p


# ---- keyswitch ------------------------------------------------------------------------------------------------------------------
def _ks_grid():
    """(kN, n, base_log, level): every accepted (B, L) with L <= 7 (all three kernels) and L = 8 ... 13 (IMAD) at kN = 2048, n + 1
    cycling through 127, 128, 129, 255, 256, 257 and 4097; a few shapes at kN = 32768 with small n (the KSK stays under 0.5 GB)"""
    shapes = [(B, L) for B in range(2, 8) for L in range(1, 14) if B * L <= 31 and (L <= 7 or B <= 3)]
    widths = [126, 127, 128, 254, 255, 256, 4096]
    out = [(2048, widths[i % len(widths)], B, L) for i, (B, L) in enumerate(shapes)]
    out += [(32768, 126, 7, 4), (32768, 128, 6, 5), (32768, 127, 4, 7), (32768, 255, 2, 13), (32768, 256, 3, 10)]
    return out


KS_GRID = _ks_grid()


def _ks_check(orc, p, ksk, x, label):
    import fhe_string_bounty_b200 as F
    kN = p.glwe_dim * p.poly_size
    need = sorted(set().union(*(probe_rows(b, kN).tolist() for b in BATCHES)))
    want = dict(zip(need, keyswitch_rows(orc, p, ksk, x[need])))
    eng = F.Engine(engine_params(p))
    eng.upload_ksk(ksk)
    kernels = (2, 1, 0) if p.ks_level <= 7 else (0,)
    for kernel in kernels:
        eng.set_tuning("ks_kernel", kernel)
        for batch in BATCHES:
            got = eng.keyswitch_batch(x[:batch])
            rows = probe_rows(batch, kN)
            bad = [int(r) for r in rows if not np.array_equal(got[r], want[int(r)])]
            assert not bad, f"{label} kN={kN} n={p.lwe_dim} B={p.ks_base_log} L={p.ks_level} ks_kernel={kernel} batch={batch}: rows {bad[:8]}"
    eng.close()
    print(f"{label} kN={kN} n={p.lwe_dim} B={p.ks_base_log} L={p.ks_level}: ks_kernel {'/'.join(map(str, kernels))}, batches {BATCHES}, "
          f"{len(need)} rows word for word")


@pytest.mark.parametrize("shape", KS_GRID, ids=[f"kN{s[0]}_n{s[1]}_B{s[2]}_L{s[3]}" for s in KS_GRID])
def test_keyswitch_range(orc, shape):
    kN, n, B, L = shape
    p = _params(orc, kN, 1, n, B, L)
    rng = np.random.default_rng(kN + 17 * n + 7 * L + B)
    ksk = rng.integers(0, 2**64, size=kN * L * (n + 1), dtype=np.uint64)
    _ks_check(orc, p, ksk, ks_inputs(p, rng, max(BATCHES)), "uniform key")


def largest_plane_sum(orc, kN, B, L):
    """the tensor-core plane sum S_p of an all-0xFF key and inputs at max_digit_word: 255 * kN * sum of the biased digits d + B/2"""
    d = orc.decompose(max_digit_word(B, L), B, L)
    return 255 * kN * sum(v + (1 << (B - 1)) for v in d)


@pytest.mark.parametrize("shape", [(32768, 126, 7, 4), (32768, 128, 6, 5)], ids=["kN32768_B7_L4", "kN32768_B6_L5"])
def test_keyswitch_plane_sums_past_2_31(orc, shape):
    """every key byte 0xFF and every mask word at the largest digits: the s32 plane sums lie between 2^31 and 2^32, and the epilogues
    read them as u32"""
    kN, n, B, L = shape
    s = largest_plane_sum(orc, kN, B, L)
    print(f"kN={kN} B={B} L={L}: largest plane sum {s} = 2^{np.log2(s):.3f}")
    assert 2**31 < s < 2**32, s
    p = _params(orc, kN, 1, n, B, L)
    ksk = np.full(kN * L * (n + 1), 2**64 - 1, dtype=np.uint64)
    x = ks_inputs(p, np.random.default_rng(9), max(BATCHES))
    x[:, :kN] = max_digit_word(B, L)
    _ks_check(orc, p, ksk, x, "all-0xFF key")


@pytest.mark.parametrize("n", [741, 742, 745, 1024])
def test_fused_ks_pbs_range(orc, n):
    """ks_pbs_batch on the tuned shape (the keyswitch epilogue hands pbs_v4 / pbs_v8 the u16 modulus switch, rows of n + 1 u16) with a
    uniform KSK and the lattice BSK, on ks_kernel 2 and 1 == orc_keyswitch followed by the exact rotation"""
    import fhe_string_bounty_b200 as F
    sms = _sms()
    p = _params(orc, 2048, 1, n, 3, 5, pbs_base_log=23, pbs_level=1)
    s = lattice_shift(p)
    rng = np.random.default_rng(0xF500 + n)
    ksk = rng.integers(0, 2**64, size=p.big_dim * p.ks_level * (n + 1), dtype=np.uint64)
    bsk = lattice_bsk(orc, p, 0xF501 + n)
    luts = lattice_luts(p, 3, 0xF502 + n)
    pool = rng.integers(0, 2**64, size=(POOL, p.big_dim + 1), dtype=np.uint64)
    small = keyswitch_rows(orc, p, ksk, pool)
    pidx = (np.arange(POOL) % 3).astype(np.uint32)
    exact = exact_unique(orc, p, bsk, small, luts, pidx)
    eng = F.Engine(engine_params(p))
    eng.upload_ksk(ksk)
    eng.upload_bsk_std(bsk)
    eng.upload_luts(luts)
    for kernel in (2, 1):
        eng.set_tuning("ks_kernel", kernel)
        for batch in (4 * sms + 3, 37):        # wide pbs_v4<4> + v8 tail, and a narrow level on the v8x2 cluster instance
            sel = np.arange(batch) % POOL
            got = eng.ks_pbs_batch(pool[sel], pidx[sel])
            assert np.array_equal(eng.keyswitch_batch(pool[sel]), small[sel]), (kernel, batch)
            assert_on_lattice(got, exact[sel], s, f"fused KS (ks_kernel {kernel}) -> PBS, n={n} [batch {batch}]")
    eng.close()


# ---- blind rotation -------------------------------------------------------------------------------------------------------------
class Case:
    """lattice BSK, LUTs and a pool of distinct inputs at one point; the exact reference once per pool row"""

    def __init__(self, orc, pt: Point, pool=POOL):
        self.orc, self.pt = orc, pt
        self.p = p = pt.params(orc)
        self.s = lattice_shift(p)
        seed = 0xA000 + 16 * pt.n + pt.B + 100 * pt.l + 1000 * pt.g
        self.bsk = lattice_bsk(orc, p, seed, nnz=pt.nnz, cmax=pt.cmax)
        self.luts = lattice_luts(p, 3, seed + 1)
        self.small = lattice_inputs(p, pool, seed + 2)
        self.idx = (np.arange(pool) % 3).astype(np.uint32)
        self.exact = exact_unique(orc, p, self.bsk, self.small, self.luts, self.idx)

    def engine(self, env=None):
        import fhe_string_bounty_b200 as F
        with _env(**(env or {})):
            e = F.Engine(engine_params(self.p))
        e.upload_bsk_std(self.bsk)
        e.upload_luts(self.luts)
        return e

    def check(self, eng, batch, label, start=3):
        """rows start, start + 1, ... of the pool (cyclically): a batch of one takes row 3, a random mask; wider batches hold the
        all-zero, all-tie and fixed-edge rows 0 ... 2 as well"""
        sel = (start + np.arange(batch)) % len(self.small)
        small, idx = self.small[sel], self.idx[sel]
        got = eng.pbs_batch(small, idx)
        return assert_on_lattice(
            got, self.exact[sel], self.s, f"{label} [{self.pt.id}, batch {batch}]",
            run_rows=lambda k, r: eng.pbs_batch(small, idx, n_iters=k)[r],
            ref_rows=lambda k, r: self.orc.pbs_exact_batch(self.p, self.bsk, small[r], self.luts, idx[r], max_steps=k),
            n_steps=pbs_steps(self.p))


def _run_tuned(case, configs, defaults):
    """configs of (label, batch, tuning) on one context (tuning reset to `defaults` after each)"""
    eng = case.engine()
    for label, batch, tuning in configs:
        for k, v in tuning.items():
            eng.set_tuning(k, v)
        case.check(eng, batch, label, start=3 if batch == 1 else 0)
        for k in tuning:
            eng.set_tuning(k, defaults[k])
    eng.close()


@pytest.mark.parametrize("pt", CLASSIC, ids=[pt.id for pt in CLASSIC])
def test_rotation_classic(orc, pt):
    sms = _sms()
    case = Case(orc, pt)
    _run_tuned(case, [
        ("pbs_classic_kernel_v4<4> + v8 tail", 4 * sms + 3, {}),
        ("pbs_classic_kernel_v4<3>", 3 * sms - 1, {}),
        ("planned cut: two waves of <3> in one launch", 4 * sms + 200, {}),
        ("planned cut: <3> wave + v8 tail", 5 * sms, {}),
        ("pbs_classic_kernel_v4<2>", 2 * sms - 1, {"narrow_kernel": 0}),
        ("pbs_classic_kernel_v4<1>", sms - 1, {"narrow_kernel": 0}),
        ("pbs_classic_kernel_v8 (one SM)", 37, {"narrow_cluster": 0}),
        ("pbs_classic_kernel_v8 (one SM, 2 per SM)", 2 * sms - 3, {"narrow_cluster": 0}),
        ("pbs_classic_kernel_v8x2 (two-SM cluster)", 37, {}),
        ("batch of one", 1, {}),
    ], defaults={"narrow_kernel": 8, "narrow_cluster": 1})
    eng = case.engine(env={"TFHE_B200_PBS_KERNEL": "generic"})
    case.check(eng, 37, "pbs_generic")
    eng.close()


@pytest.mark.parametrize("pt", MULTIBIT, ids=[pt.id for pt in MULTIBIT])
def test_rotation_multibit(orc, pt):
    sms = _sms()
    case = Case(orc, pt)
    _run_tuned(case, [
        ("pbs_multibit_kernel_v4<3> + v8 tail", 3 * sms + 2, {}),
        ("pbs_multibit_kernel_v4<2>", 2 * sms - 1, {"narrow_kernel": 0}),
        ("pbs_multibit_kernel_v4<1>", sms - 1, {"narrow_kernel": 0}),
        ("pbs_multibit_kernel_v8 (one SM)", 37, {"narrow_cluster": 0}),
        ("pbs_multibit_kernel_v8x2 (two-SM cluster)", 37, {}),
        ("batch of one", 1, {}),
    ], defaults={"narrow_kernel": 8, "narrow_cluster": 1})
    eng = case.engine(env={"TFHE_B200_PBS_KERNEL": "generic"})
    case.check(eng, 37, "pbs_generic")
    eng.close()


@pytest.mark.parametrize("pt", N512, ids=[pt.id for pt in N512])
def test_rotation_n512(orc, pt):
    sms = _sms()
    case = Case(orc, pt)
    _run_tuned(case, [
        ("pbs_n512_kernel<1>", 3, {"tuned512_min": 1}),
        ("pbs_n512_kernel<4>", sms + 5, {"tuned512_min": 1}),
        ("pbs_n512_kernel<8>", 8 * sms + 5, {"tuned512_min": 1}),
        ("pbs_generic (below tuned512_min)", 37, {}),
    ], defaults={"tuned512_min": 0})


@pytest.mark.parametrize("pt", N8192, ids=[pt.id for pt in N8192])
def test_rotation_n8192(orc, pt):
    """pbs_n8192 (one ciphertext per two-SM cluster) while 2 B <= 31, and pbs_generic; above, the tuned kernel must not be selectable
    and the default context runs pbs_generic"""
    from fhe_string_bounty_b200._native import NativeError
    sms = _sms()
    case = Case(orc, pt, pool=11)           # one ciphertext per cluster: no CTA holds two rows
    eng = case.engine()
    if 2 * pt.B <= 31:
        eng.set_tuning("tuned8192", 1)
        for batch in (3, sms // 2 + 7):
            case.check(eng, batch, "pbs_n8192")
        eng.set_tuning("tuned8192", 0)
        case.check(eng, 3, "pbs_generic")
    else:
        for batch in (3, sms // 2 + 7):
            case.check(eng, batch, "default kernel (pbs_generic)")
        with pytest.raises(NativeError, match="tuned8192"):
            eng.set_tuning("tuned8192", 1)
    eng.close()


@pytest.mark.parametrize("pt", GENERIC, ids=[pt.id for pt in GENERIC])
def test_rotation_generic(orc, pt):
    case = Case(orc, pt)
    eng = case.engine()
    case.check(eng, 37, "pbs_generic")
    eng.close()


# ---- contexts -------------------------------------------------------------------------------------------------------------------
def test_later_context_keeps_imad_keyswitch(orc):
    """context A (2_2, 5 levels) on the IMAD keyswitch, then context B with 2 levels, kept alive: both keyswitch word for word"""
    import fhe_string_bounty_b200 as F
    rng = np.random.default_rng(0xF600)
    pa = orc.params("2_2")
    pb = orc.params("2_2")
    pb.ks_base_log, pb.ks_level = 7, 2
    keys, engs, xs = [], [], []
    for p in (pa, pb):
        ksk = rng.integers(0, 2**64, size=p.big_dim * p.ks_level * (p.lwe_dim + 1), dtype=np.uint64)
        e = F.Engine(engine_params(p))
        e.set_tuning("ks_kernel", 0)
        e.upload_ksk(ksk)
        keys.append(ksk)
        engs.append(e)
        xs.append(ks_inputs(p, rng, 130))
    for p, ksk, e, x, label in zip((pa, pb), keys, engs, xs, ("A (L = 5)", "B (L = 2)")):
        got = e.keyswitch_batch(x)
        assert np.array_equal(got, keyswitch_rows(orc, p, ksk, x)), label
        print(f"context {label}, IMAD keyswitch after both were created: 130 rows word for word")
    for e in engs:
        e.close()


@pytest.mark.parametrize("level", [14, 15])
def test_keyswitch_levels_past_shared_memory_refused(orc, level):
    """(B, L) = (2, 14) and (2, 15) pass B * L <= 31 but the IMAD kernel's two stages of 8 * L key rows exceed 227 KB"""
    import fhe_string_bounty_b200 as F
    from fhe_string_bounty_b200._native import NativeError
    p = _params(orc, 2048, 1, 742, 2, level, pbs_base_log=23, pbs_level=1)
    with pytest.raises(NativeError, match="at most 13 levels"):
        F.Engine(engine_params(p))
