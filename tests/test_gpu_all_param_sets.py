"""Kernel shapes of the 36 classic PARAM_MESSAGE_<m>_CARRY_<c>_KS_PBS sets that the other GPU tests never run (run with -m gpu).

  * keyswitch: every distinct (k N, n, ks_base_log, ks_level) of the 36 sets on each of ks_kernel 2 (tcgen05), 1 (mma.sync) and 0 (IMAD),
    word for word against orc_keyswitch, on a uniform-random key and on a key of all-0xFF bytes (the u8 x u8 -> s32 exactness bound of
    keyswitch_tc.cu) with the largest digits the decomposition produces;
  * blind rotation: the lattice-key word-exact test (test_gpu_exact_rotation.py) for 3 PBS levels at N = 16384 and 32768
    (pbs_generic launch_big<14> / <15>) and one level at N = 8192 on pbs_generic; the CPU premise check for the same shapes;
  * precision: one CMUX with a dense uniform-random GGSW against the exact external product (DESIGN section 4: 2^44);
  * host programs on ciphertexts whose propagation the host layer used to get wrong (2_2 and 3_3 at degree 2m - 1, one-bit blocks on 1_3).

Only keys that are not encryptions are built from the engine's parameter table (_native.classic_params): no noise parameter is needed."""
import ctypes as C

import numpy as np
import pytest

from fhe_string_bounty_b200 import _native as N
from helpers import assert_on_lattice, engine_params, lattice_bsk, lattice_inputs, lattice_luts, lattice_shift, max_residual, pbs_steps


def oracle_params(orc, name):
    """orc.Params of any classic set from the engine's table; the noise fields stay 0 (these tests never encrypt with them)"""
    p = orc.Params()
    for k, v in N.classic_params(name).items():
        setattr(p, k, v)
    return p


def ks_shapes():
    """distinct keyswitch shapes (k N, n, base_log, level) -> the first set that has it"""
    out = {}
    for name in N._CLASSIC_SETS:
        q = N.classic_params(name)
        out.setdefault((q["glwe_dim"] * q["poly_size"], q["lwe_dim"], q["ks_base_log"], q["ks_level"]), name)
    return out


KS_SHAPES = ks_shapes()
BATCHES = (1, 127, 128, 129, 300)


def max_digit_word(B, L):
    """the word whose signed decomposition has the largest digits: +B/2 at the top level and B/2 - 1 below (d' = B, B - 1, ...).  Every
    digit at +B/2 is not reachable: a digit of B/2 stays positive only if the next level's raw digit is below B/2."""
    d = [1 << (B - 1)] + [(1 << (B - 1)) - 1] * (L - 1)
    return sum(v << (64 - (j + 1) * B) for j, v in enumerate(d)) % 2**64


def ks_inputs(p, rng, rows):
    """rows x (k N + 1): 0, 2^64 - 1, 2^63, rounding ties at 2^(63 - B L) under random upper bits, the largest digits, and random words;
    bodies random"""
    kN, B, L = p.glwe_dim * p.poly_size, p.ks_base_log, p.ks_level
    x = rng.integers(0, 2**64, size=(rows, kN + 1), dtype=np.uint64)
    tie = lambda n: (rng.integers(0, 2**(B * L), size=n, dtype=np.uint64) << np.uint64(64 - B * L)) | np.uint64(1 << (63 - B * L))
    fixed = [np.zeros(kN, np.uint64), np.full(kN, 2**64 - 1, np.uint64), np.full(kN, 2**63, np.uint64), tie(kN),
             np.full(kN, max_digit_word(B, L), np.uint64)]
    for i, f in enumerate(fixed):
        x[i, :kN] = f
    edge = np.array([0, 2**64 - 1, 2**63, max_digit_word(B, L)], dtype=np.uint64)
    pick = rng.random((rows, kN)) < 0.25
    x[:, :kN][pick] = np.where(rng.random(int(pick.sum())) < 0.5, edge[rng.integers(0, 4, int(pick.sum()))], tie(int(pick.sum())))
    x[: len(fixed), :kN] = np.stack(fixed)
    return x


def probe_rows(batch, kN):
    """every row up to kN = 4096; above it the first and last row of each 128-row tile and the batch's last row"""
    if kN <= 4096:
        return np.arange(batch)
    return np.array(sorted({r for t in range(0, batch, 128) for r in (t, min(t + 127, batch - 1))} | {batch - 1}))


def orc_keyswitch(orc, p, ksk, rows):
    out = np.zeros((len(rows), p.lwe_dim + 1), dtype=np.uint64)
    for i, r in enumerate(rows):
        orc.lib().orc_keyswitch(C.byref(p), ksk, np.ascontiguousarray(r), out[i])
    return out


def _check_keyswitch(orc, name, ksk, x, label):
    import fhe_string_bounty_b200 as F
    p = oracle_params(orc, name)
    kN = p.glwe_dim * p.poly_size
    need = sorted(set().union(*(probe_rows(b, kN).tolist() for b in BATCHES)))
    want = dict(zip(need, orc_keyswitch(orc, p, ksk, x[need])))
    eng = F.Engine(engine_params(p))
    eng.upload_ksk(ksk)                       # default ks_kernel 2: the byte planes of kernels 1 and 2 are built at upload
    for kernel in (2, 1, 0):
        eng.set_tuning("ks_kernel", kernel)
        for batch in BATCHES:
            got = eng.keyswitch_batch(x[:batch])
            rows = probe_rows(batch, kN)
            bad = [int(r) for r in rows if not np.array_equal(got[r], want[int(r)])]
            assert not bad, f"{label} {name} kN={kN} n={p.lwe_dim} B={p.ks_base_log} l={p.ks_level} ks_kernel={kernel} batch={batch}: rows {bad[:8]}"
    eng.close()
    print(f"{label} {name} (kN={kN}, n={p.lwe_dim}, B={p.ks_base_log}, l={p.ks_level}): ks_kernel 2/1/0, batches {BATCHES}, "
          f"{len(need)} rows word for word")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(KS_SHAPES), ids=[f"kN{s[0]}_n{s[1]}_B{s[2]}_l{s[3]}" for s in KS_SHAPES])
def test_keyswitch_every_shape_every_kernel(orc, shape):
    name = KS_SHAPES[shape]
    p = oracle_params(orc, name)
    rng = np.random.default_rng(shape[0] + shape[1] + 7 * shape[3])
    ksk = rng.integers(0, 2**64, size=p.glwe_dim * p.poly_size * p.ks_level * (p.lwe_dim + 1), dtype=np.uint64)
    _check_keyswitch(orc, name, ksk, ks_inputs(p, rng, max(BATCHES)), "uniform key")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["2_2", "6_0", "8_0"])
def test_keyswitch_all_ff_key(orc, name):
    """every key byte 0xFF and every input word at the largest digits: the s32 accumulator of the tensor-core kernels reaches its
    largest value (keyswitch_tc.cu: K * B * 255 < 2^31)"""
    p = oracle_params(orc, name)
    ksk = np.full(p.glwe_dim * p.poly_size * p.ks_level * (p.lwe_dim + 1), 2**64 - 1, dtype=np.uint64)
    x = ks_inputs(p, np.random.default_rng(5), max(BATCHES))
    x[:, : p.glwe_dim * p.poly_size] = max_digit_word(p.ks_base_log, p.ks_level)
    _check_keyswitch(orc, name, ksk, x, "all-0xFF key")


# ---- blind rotation on the shapes no other test runs ---------------------------------------------------------------------------
# 1_6: 3 levels (base 11), N = 16384, launch_big<14>; 1_7 / 2_6 / 3_5: 3 levels, N = 32768, launch_big<15>; 5_1 / 6_0: one level at
# N = 8192 on pbs_generic (pbs_n8192.cu takes two levels only).  A 3-level N = 32768 BSK is 3.2 GB of u64; the lattice key is written
# at 8 positions per polynomial into np.zeros, so only the touched pages are resident.
ROTATION_SETS = ["1_6", "1_7", "2_6", "3_5", "5_1", "6_0"]


def _rows(p):
    return 6 if p.poly_size <= 8192 else 3


@pytest.mark.parametrize("name", ROTATION_SETS)
def test_lattice_premise_new_shapes(orc, name):
    """CPU: the oracle's f64 PBS rounded to 2^s equals the exact PBS on these shapes (test_oracle_exact_rotation.py's premise)"""
    p = oracle_params(orc, name)
    s = lattice_shift(p)
    bsk = lattice_bsk(orc, p, seed=41, nnz=8)
    luts = lattice_luts(p, 2, seed=42)
    small = lattice_inputs(p, 2, seed=43)
    idx = np.array([0, 1], dtype=np.uint32)
    exact = orc.pbs_exact_batch(p, bsk, small, luts, idx)
    got = orc.pbs_f64_batch(p, orc.FourierKey(p, bsk), small, luts, idx)
    assert_on_lattice(got, exact, s, f"oracle f64 {name} (N={p.poly_size} l={p.pbs_level} B={p.pbs_base_log})")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ROTATION_SETS)
def test_lattice_rotation_new_shapes(orc, name):
    """pbs_generic on the shape, word for word after the full rotation; residual printed, bound 2^(s-4) (s = 31 for the 3-level sets)"""
    import fhe_string_bounty_b200 as F
    p = oracle_params(orc, name)
    s = lattice_shift(p)
    rows = _rows(p)
    bsk = lattice_bsk(orc, p, seed=0xF100, nnz=8)
    luts = lattice_luts(p, 3, seed=0xF101)
    small = lattice_inputs(p, rows, seed=0xF102)
    idx = (np.arange(rows) % 3).astype(np.uint32)
    exact = orc.pbs_exact_batch(p, bsk, small, luts, idx)
    eng = F.Engine(engine_params(p))
    eng.upload_bsk_std(bsk)
    eng.upload_luts(luts)
    got = eng.pbs_batch(small, idx)
    assert_on_lattice(got, exact, s, f"pbs_generic {name} (N={p.poly_size} l={p.pbs_level} B={p.pbs_base_log})",
                      run_rows=lambda k, r: eng.pbs_batch(small, idx, n_iters=k)[r],
                      ref_rows=lambda k, r: orc.pbs_exact_batch(p, bsk, small[r], luts, idx[r], max_steps=k), n_steps=pbs_steps(p))
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["1_7", "5_1"])
def test_dense_cmux_precision(orc, name):
    """one CMUX with a dense uniform-random GGSW at index j (every other GGSW zero, every other mask element zero) against the exact
    external product: |gpu - exact| <= 2^44 (DESIGN section 4), printed next to the oracle f64's own distance"""
    import fhe_string_bounty_b200 as F
    p = oracle_params(orc, name)
    n, N_, k1, L = p.lwe_dim, p.poly_size, p.glwe_dim + 1, p.pbs_level
    ggsw = L * k1 * k1 * N_
    rng = np.random.default_rng(0xF200)
    js = [0, n - 1]
    bsk = np.zeros(n * ggsw, dtype=np.uint64)
    for j in js:
        bsk[j * ggsw:(j + 1) * ggsw] = rng.integers(0, 2**64, size=ggsw, dtype=np.uint64)
    luts = rng.integers(0, 2**64, size=(1, p.lut_len), dtype=np.uint64)
    small = np.zeros((len(js), n + 1), dtype=np.uint64)
    for u, j in enumerate(js):
        small[u, j] = rng.integers(1, 2**64, dtype=np.uint64)
        small[u, n] = rng.integers(0, 2**64, dtype=np.uint64)
    idx = np.zeros(len(js), dtype=np.uint32)
    exact = orc.pbs_exact_batch(p, bsk, small, luts, idx)
    d_orc = max_residual(orc.pbs_f64_batch(p, orc.FourierKey(p, bsk), small, luts, idx), exact)
    eng = F.Engine(engine_params(p))
    eng.upload_bsk_std(bsk)
    eng.upload_luts(luts)
    got = eng.pbs_batch(small, idx)
    eng.close()
    d = max_residual(got, exact)
    print(f"pbs_generic {name} (N={N_} l={L} B={p.pbs_base_log}): one dense CMUX at j in {js}: max |gpu - exact| 2^{np.log2(max(d, 1)):.1f}, "
          f"oracle f64 - exact 2^{np.log2(max(d_orc, 1)):.1f} (bound 2^44)")
    assert d <= 2**44, (name, np.log2(d))


# ---- host programs on real ciphertexts --------------------------------------------------------------------------------------------
def _engine_for(keys):
    import fhe_string_bounty_b200 as F
    p, ck, sk = keys
    eng = F.Engine(engine_params(p))
    eng.upload_ksk(sk.ksk)
    eng.upload_bsk_std(sk.bsk)
    return eng


def _run_gpu(eng, keys, op, args, blocks):
    from fhe_string_bounty_b200.host import Program
    p, ck, sk = keys
    P = Program(op, args, params=engine_params(p))
    out = P.run(eng, np.stack([ck.encrypt_with_carry(int(b)) for b in blocks]))
    return [ck.decrypt_message_and_carry(c) for c in out]


@pytest.mark.gpu
def test_propagation_fixes_on_ciphertexts_2_2(keys_2_2):
    """2_2: blocks of degree 7 = 2m - 1 (the value 147 = 19 mod 64 = [3, 0, 1])"""
    eng = _engine_for(keys_2_2)
    assert _run_gpu(eng, keys_2_2, "radix_full_propagate", (3, 7), [7, 7, 7]) == [3, 0, 1]
    assert _run_gpu(eng, keys_2_2, "radix_full_propagate", (3, 7), [7, 0, 7]) == [3, 1, 3]            # 7 + 112 = 119 = 55 mod 64
    assert _run_gpu(eng, keys_2_2, "radix_default_eq", (3, 7), [7, 7, 7, 3, 0, 1]) == [1]
    assert _run_gpu(eng, keys_2_2, "radix_default_eq", (3, 7), [7, 7, 7, 3, 0, 0]) == [0]
    assert _run_gpu(eng, keys_2_2, "radix_default_lt", (3, 7), [7, 7, 7, 0, 1, 1]) == [1]             # 19 < 20
    assert _run_gpu(eng, keys_2_2, "radix_default_lt", (3, 7), [7, 7, 7, 3, 0, 1]) == [0]
    eng.close()


@pytest.mark.gpu
def test_one_bit_add_on_ciphertexts_1_3(orc):
    """1_3 (N = 2048, k = 1, one level: the tuned kernels): radix_add on one-bit blocks, whose carry states need the cur * 3 + prev packing"""
    p = orc.params("1_3")
    ck = orc.ClientKey(p, 0xF300)
    keys = (p, ck, orc.ServerKey(ck, 0xF301, fourier=False))
    eng = _engine_for(keys)
    for x, y in ((7, 1), (31, 0), (31, 1), (21, 10), (0, 0)):
        bits = lambda v: [(v >> i) & 1 for i in range(5)]
        assert _run_gpu(eng, keys, "radix_add", (5,), bits(x) + bits(y)) == bits((x + y) % 32), (x, y)
    eng.close()


@pytest.mark.gpu
def test_propagation_fixes_on_ciphertexts_3_3(orc):
    """3_3 (N = 8192, two levels: pbs_n8192.cu): blocks of degree 15 = 2m - 1"""
    p = orc.params("3_3")
    ck = orc.ClientKey(p, 0xF400)
    keys = (p, ck, orc.ServerKey(ck, 0xF401, fourier=False))
    eng = _engine_for(keys)
    assert _run_gpu(eng, keys, "radix_full_propagate", (3, 15), [15, 15, 15]) == [7, 0, 1]            # 15 * 73 = 1095 = 71 mod 512
    assert _run_gpu(eng, keys, "radix_default_eq", (3, 15), [15, 15, 15, 7, 0, 1]) == [1]
    eng.close()
