"""Many-LUT PBS on the GPU (run with -m gpu).

Every kernel instance, lattice-valued test keys (as test_gpu_exact_rotation.py), tables of F = 2, 3, 4 functions mixed in one batch:
(a) row f = 0 of every ciphertext equals, word for word, pbs_batch with the same accumulators uploaded as single-function tables;
(b) the mask words of row f equal the extraction at t_f = f * chunk * box of the mask polynomial that row 0 was extracted from, and the
    rows past a table's F are zero;
(c) on probe ciphertexts (first and last CTAs and one in between), every word of every row, body included, rounded to 2^s equals the
    extraction at t_f of the exact GLWE (tests/many_lut_ref.exact_glwe_batch, checked against orc_pbs_exact_batch at t = 0); a mismatch
    is bisected over n_iters to the first failing step.  Each case asserts, by name from torch.profiler, that the kernel instance it is
    about ran;
(c) with real 2_2 keys every function decrypts to f_f(x) for all x < chunk, through the host and device entries, the fused keyswitch and
    a 2^32 ciphertext modulus; the single-function entries refuse to run while a many-LUT table is uploaded.
"""
import re

import numpy as np
import pytest

from helpers import assert_on_lattice, engine_params, lattice_bsk, lattice_inputs, lattice_luts, lattice_shift, pbs_steps
from many_lut_ref import exact_glwe_batch, extract_at, extract_mask_at, extraction_step, mask_from_row0

pytestmark = pytest.mark.gpu


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _engine(p, bsk, env=None, tuning=None):
    import os
    import fhe_string_bounty_b200 as F
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update({k: str(v) for k, v in (env or {}).items()})
    try:
        e = F.Engine(engine_params(p))
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    e.upload_bsk_std(bsk)
    for k, v in (tuning or {}).items():
        e.set_tuning(k, v)
    return e


def _launched_kernels(run):
    """names of the CUDA kernels that run() launches (torch.profiler, CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = run()
    return out, {e.name for e in prof.events()}


def _ran(kernel, names):
    """kernel = "base" or "base<CTS>": demangled or mangled names; an untemplated base must not match its x2 sibling"""
    if "<" in kernel:
        base, cts = kernel[:-1].split("<")
        pat = re.escape(base) + rf"(<{cts}>|ILi{cts}E)"
    else:
        pat = re.escape(kernel) + r"(\(|<|E|I|$)"
    return any(re.search(pat, n) for n in names)


def _probe_rows(batch, count=8):
    if batch <= count:
        return list(range(batch))
    return sorted({0, 1, 2, 3, batch // 2, batch - 3, batch - 2, batch - 1})[:count]


def _check_instance(orc, name, batch, label, kernel, env=None, tuning=None, nnz=8, probes=8):
    p = orc.params(name)
    total = p.msg_mod * p.carry_mod
    fcounts = np.array([F for F in (2, 3, 4) if F <= total], dtype=np.uint32)
    s = lattice_shift(p)
    bsk = lattice_bsk(orc, p, 0xA100, nnz=nnz)
    accs = lattice_luts(p, len(fcounts), 0xA101)
    small = lattice_inputs(p, batch, 0xA102)
    idx = ((np.arange(batch) * 7 + np.arange(batch) // 64) % len(fcounts)).astype(np.uint32)
    eng = _engine(p, bsk, env, tuning)
    eng.upload_luts(accs)
    single = eng.pbs_batch(small, idx)
    eng.upload_many_luts(accs, fcounts)
    rows, names = _launched_kernels(lambda: eng.pbs_many_batch(small, idx))
    assert _ran(kernel, names), f"{label} [{name}, batch {batch}]: {kernel} did not run; launched {sorted(names)}"
    S = int(fcounts.max())
    assert rows.shape == (batch, S, p.big_dim + 1)
    # (a) row 0 is the single-function PBS, every row of the batch
    bad = np.flatnonzero((rows[:, 0] != single).any(axis=1))
    assert bad.size == 0, f"{label} [{name}, batch {batch}]: row 0 differs from pbs_batch at ciphertexts {bad[:8]}"
    # (b) the mask words of every row f > 0 of every ciphertext are the extraction at t_f of the mask row 0 came from
    kN = p.glwe_dim * p.poly_size
    for i in range(batch):
        A = mask_from_row0(p, rows[i, 0])
        F = int(fcounts[idx[i]])
        for f in range(1, F):
            want = extract_mask_at(A, f * extraction_step(p, F))
            assert np.array_equal(rows[i, f, :kN], want), f"{label} [{name}, batch {batch}]: ciphertext {i}, function {f} of {F}"
        assert not rows[i, F:].any(), f"{label}: rows past F of ciphertext {i} are not zero"
    # (c) whole rows, body included, of the probe ciphertexts against the extractions of the exact GLWE, rounded to 2^s; a mismatch is
    # bisected over n_iters
    pr = _probe_rows(batch, probes)
    pairs = [(i, f) for i in pr for f in range(int(fcounts[idx[i]]))]

    def run_rows(out, sel):
        return np.stack([out[pairs[r][0], pairs[r][1]] for r in sel])

    def ref(k, sel):
        g = exact_glwe_batch(p, bsk, small[pr], accs, idx[pr], max_steps=k)
        return np.stack([extract_at(g[pr.index(pairs[r][0])][None], pairs[r][1] * extraction_step(p, int(fcounts[idx[pairs[r][0]]])))[0]
                         for r in sel])

    got = run_rows(rows, range(len(pairs)))
    exact = ref(None, range(len(pairs)))
    assert_on_lattice(got, exact, s, f"{label} [{name}, batch {batch}], {len(pairs)} probe rows of {len(pr)} ciphertexts",
                      run_rows=lambda k, sel: run_rows(eng.pbs_many_batch(small, idx, n_iters=k), sel), ref_rows=ref, n_steps=pbs_steps(p))
    eng.close()
    print(f"{label} [{name}, batch {batch}]: {kernel} ran; {int(fcounts[idx].sum())} rows, row 0 == pbs_batch, masks of rows f > 0 exact")


def _classic_configs(sms):
    return [
        ("pbs_classic_kernel_v4<4> + v8 tail", "pbs_classic_kernel_v4<4>", 4 * sms + 3, {}, {}),
        ("pbs_classic_kernel_v4<3>", "pbs_classic_kernel_v4<3>", 3 * sms - 1, {}, {}),
        ("pbs_classic_kernel_v4<2>", "pbs_classic_kernel_v4<2>", 2 * sms - 1, {}, {"narrow_kernel": 0}),
        ("pbs_classic_kernel_v4<1>", "pbs_classic_kernel_v4<1>", sms - 1, {}, {"narrow_kernel": 0}),
        ("pbs_classic_kernel_v8 (one SM, 2 per SM)", "pbs_classic_kernel_v8<2>", 2 * sms - 3, {}, {"narrow_cluster": 0}),
        ("pbs_classic_kernel_v8 (one SM)", "pbs_classic_kernel_v8<1>", 37, {}, {"narrow_cluster": 0}),
        ("pbs_classic_kernel_v8x2 (two-SM cluster)", "pbs_classic_kernel_v8x2", 37, {}, {}),
        ("pbs_generic", "pbs_generic_kernel", 37, {"TFHE_B200_PBS_KERNEL": "generic"}, {}),
    ]


def test_classic_2_2_every_instance(orc):
    for label, kernel, batch, env, tuning in _classic_configs(_sms()):
        _check_instance(orc, "2_2", batch, label, kernel, env, tuning)


def test_multibit_2_2_g3_every_instance(orc):
    sms = _sms()
    for label, kernel, batch, tuning in (("pbs_multibit_kernel_v4<3> + v8 tail", "pbs_multibit_kernel_v4<3>", 3 * sms + 2, {}),
                                         ("pbs_multibit_kernel_v4<2>", "pbs_multibit_kernel_v4<2>", 2 * sms - 1, {"narrow_kernel": 0}),
                                         ("pbs_multibit_kernel_v4<1>", "pbs_multibit_kernel_v4<1>", sms - 1, {"narrow_kernel": 0}),
                                         ("pbs_multibit_kernel_v8 (one SM)", "pbs_multibit_kernel_v8", 37, {"narrow_cluster": 0}),
                                         ("pbs_multibit_kernel_v8x2 (two-SM cluster)", "pbs_multibit_kernel_v8x2", 37, {})):
        _check_instance(orc, "multibit_2_2_g3", batch, label, kernel, tuning=tuning, nnz=4, probes=4)


def test_tuned_n512_and_n8192(orc):
    sms = _sms()
    for batch, cts in ((3, 1), (sms + 5, 4), (8 * sms + 5, 8)):
        _check_instance(orc, "1_1", batch, f"pbs_n512_kernel<{cts}>", f"pbs_n512_kernel<{cts}>", tuning={"tuned512_min": 1})
    _check_instance(orc, "3_3", sms // 2 + 7, "pbs_n8192", "pbs_n8192_kernel", tuning={"tuned8192": 1}, probes=4)


@pytest.mark.parametrize("name", ["2_3", "4_4", "multibit_2_2_g2", "multibit_1_1_g3"])
def test_generic_shapes(orc, name):
    p = orc.params(name)
    kernel = "pbs_generic_big_kernel" if p.poly_size > 8192 else "pbs_generic_kernel"
    _check_instance(orc, name, 12, "pbs_generic", kernel, nnz=8 if not p.grouping_factor else 4, probes=3 if p.poly_size > 8192 else 8)


def _fns(F, total, seed):
    rng = np.random.default_rng(seed)
    t = rng.integers(0, 16, size=(F, total))
    return [(lambda x, r=r: int(r[x])) for r in t]


def test_real_keys_decrypt_every_function(keys_2_2):
    """all x < chunk through ks_pbs_many_batch (fused keyswitch), pbs_many_batch and the two device entries, F = 2, 3, 4 mixed"""
    import torch
    import fhe_string_bounty_b200 as FB
    p, ck, sk = keys_2_2
    total = p.msg_mod * p.carry_mod
    fcounts = [2, 3, 4]
    fns = [_fns(F, total, 0xA200 + F) for F in fcounts]
    accs = np.stack([FB.many_lut_accumulator(engine_params(p), f) for f in fns])
    xs, idx = [], []
    for l, F in enumerate(fcounts):
        for x in range(total // F):
            xs.append(x)
            idx.append(l)
    reps = 5
    xs, idx = np.array(xs * reps), np.array(idx * reps, dtype=np.uint32)
    cts = ck.encrypt_batch(xs)
    small = np.stack([sk.keyswitch(c) for c in cts])
    eng = FB.Engine(engine_params(p))
    eng.upload_ksk(sk.ksk)
    eng.upload_bsk_std(sk.bsk)
    eng.upload_many_luts(accs, fcounts)
    with pytest.raises(FB.NativeError, match="many-LUT"):
        eng.pbs_batch(small, idx)
    with pytest.raises(FB.NativeError, match="many-LUT"):
        eng.ks_pbs_batch(cts, idx)
    S, L = 4, (p.big_dim + 1)
    outs = {"ks_pbs_many_batch": eng.ks_pbs_many_batch(cts, idx), "pbs_many_batch": eng.pbs_many_batch(small, idx)}
    d_out = torch.zeros((len(xs) * S * L,), dtype=torch.int64, device="cuda")
    d_idx = torch.from_numpy(idx.view(np.int32)).cuda()
    eng.ks_pbs_many_batch_device(torch.from_numpy(cts.view(np.int64)).cuda(), d_idx, d_out, len(xs))
    eng.synchronize()
    outs["ks_pbs_many_batch_device"] = d_out.cpu().numpy().view(np.uint64).reshape(len(xs), S, L)
    eng.pbs_many_batch_device(torch.from_numpy(small.view(np.int64)).cuda(), d_idx, d_out, len(xs))
    eng.synchronize()
    outs["pbs_many_batch_device"] = d_out.cpu().numpy().view(np.uint64).reshape(len(xs), S, L)
    for label, rows in outs.items():
        for i, (x, l) in enumerate(zip(xs, idx)):
            for f in range(fcounts[l]):
                got = ck.decrypt_message_and_carry(rows[i, f])
                assert got == fns[l][f](x), (label, i, int(x), int(l), f, got)
    # a 2^32 ciphertext modulus rounds every row of every function, negated words (mask words past t_f) as -round(-x)
    eng.set_ciphertext_modulus_log2(32)
    r32 = eng.pbs_many_batch(small, idx)
    eng.close()
    r64 = outs["pbs_many_batch"]
    N, shift = p.poly_size, np.uint64(31)
    for i, l in enumerate(idx):
        F = fcounts[l]
        for f in range(F):
            t = f * (total // F) * (N // total)
            neg = np.zeros(L, dtype=bool)
            neg[:L - 1] = (np.arange(L - 1) % N) > t
            x = r64[i, f].copy()
            x[neg] = np.uint64(0) - x[neg]
            x = (((x >> shift) + np.uint64(1)) & ~np.uint64(1)) << shift
            x[neg] = np.uint64(0) - x[neg]
            assert np.array_equal(r32[i, f], x), (i, f)
    print(f"real 2_2 keys: {len(xs)} ciphertexts x F in {fcounts}: every function decrypts through 4 entry points; 2^32 rounding exact")


def test_refusals(keys_2_2):
    import fhe_string_bounty_b200 as FB
    p, ck, sk = keys_2_2
    eng = FB.Engine(engine_params(p))
    acc = np.zeros((1, p.lut_len), dtype=np.uint64)
    for F in (0, 1, 17):
        with pytest.raises(FB.NativeError, match="functions"):
            eng.upload_many_luts(acc, [F])
    with pytest.raises(FB.NativeError, match="no many-LUT table"):
        eng.pbs_many_batch(np.zeros((1, p.lwe_dim + 1), dtype=np.uint64))
    eng.close()
