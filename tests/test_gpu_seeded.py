"""GPU parity for seeded (compressed) server keys: masks re-drawn on the device from the compression seed must reproduce, bit for bit, the
keys that the reference's decompression (oracle/csprng_oracle.c) produces.

The first tests load real 2_2 and multibit_2_2_g3 keys and decrypt.  The sweep below runs one parameter set per distinct (BSK shape,
KSK shape, kernel family) of the 36 classic and 6 multi-bit sets (tests/seeded_shapes.py), on keys with uniform random bodies and seeds
of varied bytes, all 0x00 and all 0xFF:
  * KSK: keyswitch_batch on every keyswitch kernel the shape allows, seeded upload == standard upload of orc_decompress_seeded_ksk on
    random inputs (a nonzero digit at every level), and == orc_keyswitch on some rows; probe rows (tests/seeded_shapes.probe_rows: CTA
    boundaries inside a row, the last word of the stream) read back directly -- an input whose only nonzero digit is +1 at (i0, j0) gives
    minus that row -- against orc_csprng_mask_words.
  * BSK: pbs_batch and pbs_many_batch on every kernel instance the set runs (pinned by batch size and set_tuning), seeded upload ==
    standard upload of orc_decompress_seeded_bsk on every word of every row.  The kernels are deterministic, so equal words mean equal
    Fourier keys in every copy finish_bsk builds.  Every shape up to N = 8192 and one 3-level set each at N = 16384 and 32768 get this
    on the whole key; the other N >= 16384 sets on probe GGSWs (an input whose mask is zero but at index j runs one CMUX with GGSW j,
    compared with a standard key that holds only the probe GGSWs).
  * bincode blobs (oracle/wire.py): load_compressed_server_key == upload_seeded_*, a blob that differs in one parameter field is
    refused, and seeded, serialized and standard uploads replace each other in one context, also while ks_kernel = 0 or tuned8192 = 0
    is selected."""
import ctypes as C
import os
import time
from contextlib import contextmanager

import numpy as np
import pytest

from helpers import engine_params, keyswitch_rows
from seeded_shapes import (PARAM_FIELDS, SHAPES, bsk_stream, full_check, kernel_family, ksk_stream, mutated_params, probe_rows, seeded_key,
                           stream_rows, zero_body_key)

pytestmark = pytest.mark.gpu


def _engines(F, p, sk_like, csk):
    ksk, bsk = csk.decompress()                      # oracle = reference algorithm on the CPU
    a = F.Engine(engine_params(p))                   # device-side decompression
    a.upload_seeded_ksk(csk.ksk_seed, csk.ksk_bodies)
    a.upload_seeded_bsk(csk.bsk_seed, csk.bsk_bodies)
    b = F.Engine(engine_params(p))                   # standard upload of the oracle-decompressed keys
    b.upload_ksk(ksk)
    b.upload_bsk_std(bsk)
    return a, b, ksk, bsk


def test_seeded_keys_2_2_bit_exact(orc, keys_2_2):
    import fhe_string_bounty_b200 as F
    p, ck, sk = keys_2_2
    csk = orc.CompressedServerKey(ck, sk, ksk_seed=0x00112233445566778899AABBCCDDEEFF, bsk_seed=0xB200B200B200B200B200B200B200B200)
    a, b, ksk, bsk = _engines(F, p, sk, csk)
    acc, _ = sk.generate_lookup_table(lambda x: (5 * x + 3) % 16)
    for e in (a, b):
        e.upload_luts(acc[None, :])
    vals = np.arange(48) % 16
    cts = ck.encrypt_batch(vals)
    ks_a, ks_b = a.keyswitch_batch(cts), b.keyswitch_batch(cts)
    # keyswitch is exact integer arithmetic over EVERY word of the key: equal outputs <=> equal keys (up to 2^-64 collisions)
    assert np.array_equal(ks_a, ks_b)
    sk2 = orc.ServerKey.__new__(orc.ServerKey)
    sk2.p, sk2.ksk, sk2.bsk, sk2._fourier = p, ksk, bsk, None
    assert np.array_equal(ks_a[:4], np.stack([sk2.keyswitch(c) for c in cts[:4]]))
    out_a, out_b = a.ks_pbs_batch(cts, None), b.ks_pbs_batch(cts, None)
    assert np.array_equal(out_a, out_b)              # same kernel, same key bits => identical ciphertexts
    assert list(ck.decrypt_batch(out_a)) == [(5 * int(v) + 3) % 16 for v in vals]
    a.close(); b.close()


def test_seeded_keys_multibit_bit_exact(orc, keys_multibit):
    import fhe_string_bounty_b200 as F
    p, ck, sk = keys_multibit
    csk = orc.CompressedServerKey(ck, sk, ksk_seed=7, bsk_seed=(1 << 127) | 12345)
    a, b, _, _ = _engines(F, p, sk, csk)
    acc, _ = sk.generate_lookup_table(lambda x: (x * x) % 16)
    for e in (a, b):
        e.upload_luts(acc[None, :])
    vals = np.arange(20) % 16
    cts = ck.encrypt_batch(vals)
    assert np.array_equal(a.keyswitch_batch(cts), b.keyswitch_batch(cts))
    out_a, out_b = a.ks_pbs_batch(cts, None), b.ks_pbs_batch(cts, None)
    assert np.array_equal(out_a, out_b)
    assert list(ck.decrypt_batch(out_a)) == [(int(v) * int(v)) % 16 for v in vals]
    a.close(); b.close()


def test_seeded_upload_errors(orc, keys_2_2):
    import fhe_string_bounty_b200 as F
    p, ck, sk = keys_2_2
    e = F.Engine(engine_params(p))
    seed = orc.seed_bytes(1)
    with pytest.raises(RuntimeError, match="seeded keyswitch key length"):
        e.upload_seeded_ksk(seed, np.zeros(17, dtype=np.uint64))
    with pytest.raises(RuntimeError, match="seeded bootstrap key length"):
        e.upload_seeded_bsk(seed, np.zeros(2048, dtype=np.uint64))
    assert e.lib.tfhe_b200_upload_seeded_ksk(e.h, None, None, 0) != 0
    e.close()


def test_load_serialized_compressed_server_key(orc, keys_2_2):
    """bincode blob -> tfhe_b200_load_compressed_server_key == upload_seeded_* with the same seeds and bodies (identical ciphertexts);
    a blob of another parameter set is refused."""
    import fhe_string_bounty_b200 as F
    from fhe_string_bounty_b200 import wire
    from oracle import wire as W
    p, ck, sk = keys_2_2
    csk = orc.CompressedServerKey(ck, sk, ksk_seed=11, bsk_seed=22)
    blob = W.serialize_compressed_server_key(csk)
    v = wire.parse_compressed_server_key(blob)
    a = F.Engine(F.Params(**{k: getattr(v.params, k) for k, _ in F.Params._fields_}))   # parameter set discovered from the blob
    a.load_compressed_server_key(blob)
    b = F.Engine(engine_params(p))
    b.upload_seeded_ksk(csk.ksk_seed, csk.ksk_bodies)
    b.upload_seeded_bsk(csk.bsk_seed, csk.bsk_bodies)
    acc, _ = sk.generate_lookup_table(lambda x: (x + 7) % 16)
    for e in (a, b):
        e.upload_luts(acc[None, :])
    vals = np.arange(16)
    cts = ck.encrypt_batch(vals)
    out_a, out_b = a.ks_pbs_batch(cts, None), b.ks_pbs_batch(cts, None)
    assert np.array_equal(out_a, out_b)
    assert list(ck.decrypt_batch(out_a)) == [(int(x) + 7) % 16 for x in vals]
    toy = orc.params("toy")
    tck = orc.ClientKey(toy, 1)
    tsk = orc.ServerKey(tck, 2, fourier=False)
    with pytest.raises(RuntimeError, match="parameter set"):
        a.load_compressed_server_key(W.serialize_compressed_server_key(orc.CompressedServerKey(tck, tsk, 1, 2)))
    a.close(); b.close()


# ---- every shape ---------------------------------------------------------------------------------------------------------------------
def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@contextmanager
def _env(**kv):
    """environment variables read at Engine creation (TFHE_B200_*)"""
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


class _Clock:
    def __init__(self, name):
        self.name, self.t = name, time.time()

    def lap(self, what):
        now = time.time()
        print(f"  [{self.name}] {what}: {now - self.t:.2f} s")
        self.t = now


def _ks_kernels(p):
    """keyswitch kernels a context of p can run, its default first (c_api.cu: tcgen05 needs k N l a multiple of 128, both tensor-core
    kernels at most 7 levels)"""
    if p.ks_level > 7:
        return [0]
    return ([2] if p.glwe_dim * p.poly_size * p.ks_level % 128 == 0 else []) + [1, 0]


def _ks_probe_inputs(p, rows):
    """row r = (input index i0, level index j0) of the KSK: the input whose only nonzero decomposition digit is +1 at level L - j0 of
    word i0 (levels stored L .. 1), body 0; its keyswitch output is minus row r, mask and body"""
    L, B = p.ks_level, p.ks_base_log
    x = np.zeros((len(rows), p.glwe_dim * p.poly_size + 1), dtype=np.uint64)
    for u, r in enumerate(rows):
        i0, j0 = divmod(int(r), L)
        x[u, i0] = np.uint64(1 << (64 - B * (L - j0)))
    return x


def _mismatch(got, want):
    return int((got != want).sum())


@pytest.mark.parametrize("name", SHAPES)
def test_seeded_ksk_every_shape(orc, name):
    import fhe_string_bounty_b200 as F
    clk = _Clock(name)
    key = seeded_key(orc, name)
    p = key.p
    n_rows, n, _ = ksk_stream(p)
    full = full_check(p, name)
    rows = probe_rows(n_rows, n)
    probe_x = _ks_probe_inputs(p, rows)
    want_probe = np.zeros((len(rows), n + 1), dtype=np.uint64)
    want_probe[:, :n] = np.uint64(0) - stream_rows(orc, key.ksk_seed, rows, n)
    want_probe[:, n] = np.uint64(0) - key.ksk_bodies[rows]
    clk.lap(f"KSK {n_rows} rows x ({n} + 1), probe rows {rows} from the stream")
    a = F.Engine(engine_params(p))
    a.upload_seeded_ksk(key.ksk_seed, key.ksk_bodies)
    clk.lap("upload_seeded_ksk")
    if full:
        ref = key.ksk()
        clk.lap("orc_decompress_seeded_ksk")
        assert np.array_equal(keyswitch_rows(orc, p, ref, probe_x), want_probe), "the probe inputs must select minus the row"
        b = F.Engine(engine_params(p))
        b.upload_ksk(ref)
        clk.lap("standard upload of the reference KSK")
        x = np.random.default_rng(0x5EED + n_rows).integers(0, 2**64, size=(129, p.glwe_dim * p.poly_size + 1), dtype=np.uint64)
        m = 16 if p.poly_size <= 8192 else 4
        want_x = keyswitch_rows(orc, p, ref, x[:m])
        del ref
        clk.lap(f"orc_keyswitch of {m} random rows")
    for kernel in _ks_kernels(p):
        a.set_tuning("ks_kernel", kernel)
        got = a.keyswitch_batch(probe_x)
        assert np.array_equal(got, want_probe), \
            f"{name} ks_kernel={kernel}: probe rows {[r for r, g, w in zip(rows, got, want_probe) if not np.array_equal(g, w)]} differ from the stream"
        msg = f"{name} ks_kernel={kernel}: probe rows {rows} word for word against orc_csprng_mask_words"
        if full:
            b.set_tuning("ks_kernel", kernel)
            ga, gb = a.keyswitch_batch(x), b.keyswitch_batch(x)
            assert _mismatch(ga, gb) == 0, f"{name} ks_kernel={kernel}: {_mismatch(ga, gb)} words differ, rows {np.flatnonzero((ga != gb).any(1))[:8]}"
            assert np.array_equal(ga[:m], want_x), f"{name} ks_kernel={kernel}: differs from orc_keyswitch"
            msg += f"; {len(x)} random rows seeded == standard upload, 0 mismatching words; {m} rows == orc_keyswitch"
        print(msg)
    clk.lap("keyswitch checks")
    a.close()
    if full:
        b.close()


def _pbs_configs(family, sms):
    """{environment: [(instance, batch, tuning)]}: every PBS kernel instance a context of the family runs"""
    if family == "classic_v4_v8":
        return {(): [("pbs_classic_kernel_v4<4> + v8 tail", 4 * sms + 3, {}),
                     ("pbs_classic_kernel_v4<3>", 3 * sms - 1, {}),
                     ("pbs_classic_kernel_v4<2>", 2 * sms - 1, {"narrow_kernel": 0}),
                     ("pbs_classic_kernel_v4<1>", sms - 1, {"narrow_kernel": 0}),
                     ("pbs_classic_kernel_v8 (one SM)", 37, {"narrow_cluster": 0}),
                     ("pbs_classic_kernel_v8x2 (two-SM cluster)", 37, {})],
                (("TFHE_B200_PBS_KERNEL", "generic"),): [("pbs_generic", 37, {})]}
    if family == "multibit_v4_v8":
        return {(): [("pbs_multibit_kernel_v4<3> + v8 tail", 3 * sms + 2, {}),
                     ("pbs_multibit_kernel_v4<2>", 2 * sms - 1, {"narrow_kernel": 0}),
                     ("pbs_multibit_kernel_v4<1>", sms - 1, {"narrow_kernel": 0}),
                     ("pbs_multibit_kernel_v8 (one SM)", 37, {"narrow_cluster": 0}),
                     ("pbs_multibit_kernel_v8x2 (two-SM cluster)", 37, {})]}
    if family == "n512":
        return {(): [("pbs_n512<1>", 3, {"tuned512_min": 1}), ("pbs_n512<4>", sms + 5, {"tuned512_min": 1}),
                     ("pbs_n512<8>", 8 * sms + 5, {"tuned512_min": 1}), ("pbs_generic (below tuned512_min)", 37, {})]}
    if family == "n8192":
        return {(): [("pbs_n8192", sms // 2 + 7, {}), ("pbs_generic (tuned8192 = 0)", 24, {"tuned8192": 0})]}
    if family.startswith("generic_big"):
        return {(): [(f"pbs_generic launch_big<{family[len('generic_big'):]}>", 4, {})]}
    return {(): [("pbs_generic", 24, {})]}


def _set_tuning(e, family, tuning):
    """the instance's tuning on top of the defaults (tuning persists on a context)"""
    base = {"narrow_kernel": 8, "narrow_cluster": 1, "tuned512_min": 0}
    if family == "n8192":
        base["tuned8192"] = 1
    for k, v in {**base, **tuning}.items():
        e.set_tuning(k, v)


def _luts(p, rng):
    import fhe_string_bounty_b200 as F
    total = p.msg_mod * p.carry_mod
    luts = rng.integers(0, 2**64, size=(3, p.lut_len), dtype=np.uint64)
    fns = np.array([2, min(3, total), 2], dtype=np.uint32)
    accs = np.stack([F.many_lut_accumulator(engine_params(p), [lambda x, a=a, f=f: (a * x + f) % total for f in range(int(F_))])
                     for a, F_ in zip((1, 3, 5), fns)])
    return luts, accs, fns


def _compare_pbs(a, b, small, idx, luts, accs, fns, label):
    """pbs_batch and pbs_many_batch on two contexts: every word of every row equal"""
    for e in (a, b):
        e.upload_luts(luts)
    ga, gb = a.pbs_batch(small, idx), b.pbs_batch(small, idx)
    bad = _mismatch(ga, gb)
    assert bad == 0, f"{label}: pbs_batch: {bad} words differ, rows {np.flatnonzero((ga != gb).any(1))[:8].tolist()}"
    assert (ga != 0).mean() > 0.9
    for e in (a, b):
        e.upload_many_luts(accs, fns)
    ma, mb = a.pbs_many_batch(small, idx), b.pbs_many_batch(small, idx)
    bad = _mismatch(ma, mb)
    assert bad == 0, f"{label}: pbs_many_batch: {bad} words differ, rows {np.flatnonzero((ma != mb).any(axis=(1, 2)))[:8].tolist()}"
    assert (ma[:, 0] != 0).mean() > 0.9
    print(f"{label}: {len(small)} rows, pbs_batch and pbs_many_batch (F = {sorted(set(fns.tolist()))}) word for word, 0 mismatching words")


def _one_cmux_inputs(p, ggsws, rng):
    """small LWEs whose mask is zero but at GGSW index j (a nonzero modulus-switched value): the blind rotation is one CMUX with GGSW j"""
    lg = int(p.poly_size).bit_length() - 1
    x = np.zeros((len(ggsws), p.lwe_dim + 1), dtype=np.uint64)
    for u, j in enumerate(ggsws):
        x[u, j] = np.uint64(int(rng.integers(1, 2 * p.poly_size)) << (63 - lg))
        x[u, p.lwe_dim] = rng.integers(0, 2**64, dtype=np.uint64)
    return x


@pytest.mark.parametrize("name", SHAPES)
def test_seeded_bsk_every_shape(orc, name):
    import fhe_string_bounty_b200 as F
    clk = _Clock(name)
    key = seeded_key(orc, name)
    p = key.p
    family = kernel_family(engine_params(p))
    n_rows, kN, N_ = bsk_stream(p)
    rng = np.random.default_rng(0xB5B + n_rows)
    luts, accs, fns = _luts(p, rng)
    sms = _sms()
    configs = _pbs_configs(family, sms)
    if full_check(p, name):
        ref = key.bsk()
        what = f"the whole key ({n_rows} GLWE rows x {kN} + {N_})"
        batch = max(b for cs in configs.values() for _, b, _ in cs)
        small = rng.integers(0, 2**64, size=(batch, p.lwe_dim + 1), dtype=np.uint64)
    else:
        # probe GGSWs: the ones holding the probe GLWE rows, and one in the middle
        per_ggsw = p.pbs_level * (p.glwe_dim + 1)
        ggsws = sorted({r // per_ggsw for r in probe_rows(n_rows, kN)} | {p.lwe_dim // 2})
        ref = np.zeros((n_rows, kN + N_), dtype=np.uint64)
        for j in ggsws:
            g = np.arange(j * per_ggsw, (j + 1) * per_ggsw)
            ref[g] = key.bsk_rows(g)
        ref = ref.ravel()
        what = f"probe GGSWs {ggsws} (GLWE rows {probe_rows(n_rows, kN)} of {n_rows})"
        small = _one_cmux_inputs(p, ggsws, rng)
        configs = {env: [(label, len(small), t) for label, _, t in cs] for env, cs in configs.items()}
    idx = rng.integers(0, 3, size=len(small)).astype(np.uint32)
    clk.lap(f"reference BSK: {what}")
    for env, cs in configs.items():
        with _env(**dict(env)):
            a, b = F.Engine(engine_params(p)), F.Engine(engine_params(p))
        a.upload_seeded_bsk(key.bsk_seed, key.bsk_bodies)
        clk.lap(f"upload_seeded_bsk{' ' + str(dict(env)) if env else ''}")
        b.upload_bsk_std(ref)
        clk.lap("standard upload of the reference BSK")
        for label, batch, tuning in cs:
            for e in (a, b):
                _set_tuning(e, family, tuning)
            _compare_pbs(a, b, small[:batch], idx[:batch], luts, accs, fns, f"{name} {label} [{what}]")
        clk.lap("PBS checks")
        a.close(); b.close()


def _blob_engine(F, blob):
    from fhe_string_bounty_b200 import wire
    v = wire.parse_compressed_server_key(blob)
    e = F.Engine(F.Params(**{k: getattr(v.params, k) for k, _ in F.Params._fields_}))   # parameter set discovered from the blob
    e.load_compressed_server_key(blob)
    return e


def _same_words(x, s, big, small, idx, luts, label):
    """keyswitch_batch and pbs_batch of context x equal those of context s, every word"""
    for e in (x, s):
        e.upload_luts(luts)
    bad_ks = _mismatch(x.keyswitch_batch(big), s.keyswitch_batch(big))
    bad_pbs = _mismatch(x.pbs_batch(small, idx), s.pbs_batch(small, idx))
    assert bad_ks == bad_pbs == 0, f"{label}: {bad_ks} keyswitch_batch words and {bad_pbs} pbs_batch words differ"


def _select_alternatives(e, p, family, on):
    """on = False: ks_kernel 0 and tuned8192 0, where the shape has them; on = True: back to the defaults"""
    ks = _ks_kernels(p)
    if len(ks) > 1:
        e.set_tuning("ks_kernel", ks[0] if on else 0)
    if family == "n8192":
        e.set_tuning("tuned8192", 1 if on else 0)


@pytest.mark.parametrize("name", SHAPES)
def test_compressed_blob_every_shape(orc, name):
    import fhe_string_bounty_b200 as F
    from oracle import wire as W
    clk = _Clock(name)
    key = seeded_key(orc, name)
    p = key.p
    family = kernel_family(engine_params(p))
    rng = np.random.default_rng(0xB10B + p.lwe_dim)
    blob = key.blob()
    clk.lap(f"blob of {len(blob)} bytes")
    s = F.Engine(engine_params(p))
    s.upload_seeded_ksk(key.ksk_seed, key.ksk_bodies)
    s.upload_seeded_bsk(key.bsk_seed, key.bsk_bodies)
    c = _blob_engine(F, blob)
    clk.lap("upload_seeded_* and load_compressed_server_key")
    rows = 24 if p.poly_size <= 8192 else 4
    big = rng.integers(0, 2**64, size=(rows, p.glwe_dim * p.poly_size + 1), dtype=np.uint64)
    small = rng.integers(0, 2**64, size=(rows, p.lwe_dim + 1), dtype=np.uint64)
    idx = rng.integers(0, 3, size=rows).astype(np.uint32)
    luts = rng.integers(0, 2**64, size=(3, p.lut_len), dtype=np.uint64)
    _same_words(c, s, big, small, idx, luts, f"{name} blob")
    clk.lap("blob == upload_seeded: keyswitch and PBS words")
    print(f"{name}: load_compressed_server_key == upload_seeded_*, {rows} rows of keyswitch_batch and pbs_batch word for word")
    if p.poly_size > 8192:
        s.close(); c.close()
        return
    for field in PARAM_FIELDS:
        other = W.serialize_compressed_server_key(zero_body_key(orc, mutated_params(orc, p, field)))
        with pytest.raises(RuntimeError, match="parameter set"):
            c.load_compressed_server_key(other)
    _same_words(c, s, big, small, idx, luts, f"{name} after the refused blobs")
    clk.lap(f"a blob differing in each of {PARAM_FIELDS} is refused, the loaded key stays")
    print(f"{name}: blobs differing in one parameter field refused ({', '.join(PARAM_FIELDS)})")
    # seeded, serialized and standard uploads replace each other in one context, with the alternative kernels selected meanwhile
    std_ksk = rng.integers(0, 2**64, size=orc.lib().orc_ksk_len(C.byref(p)), dtype=np.uint64)
    std_bsk = rng.integers(0, 2**64, size=orc.lib().orc_bsk_len(C.byref(p)), dtype=np.uint64)
    t = F.Engine(engine_params(p))
    t.upload_ksk(std_ksk)
    t.upload_bsk_std(std_bsk)
    x = _blob_engine(F, seeded_key(orc, name, variant=1).blob())
    steps = [("upload_seeded_*", lambda: (x.upload_seeded_ksk(key.ksk_seed, key.ksk_bodies), x.upload_seeded_bsk(key.bsk_seed, key.bsk_bodies)), s),
             ("upload_ksk / upload_bsk_std", lambda: (x.upload_ksk(std_ksk), x.upload_bsk_std(std_bsk)), t),
             ("load_compressed_server_key", lambda: x.load_compressed_server_key(blob), s)]
    for label, upload, want in steps:
        _select_alternatives(x, p, family, on=False)
        upload()
        _select_alternatives(x, p, family, on=True)
        _same_words(x, want, big, small, idx, luts, f"{name}: {label} replacing the previous key")
    clk.lap("replacement")
    print(f"{name}: another key's blob, then {', then '.join(l for l, _, _ in steps)} in one context (ks_kernel 0"
          f"{' and tuned8192 0' if family == 'n8192' else ''} selected during each upload): the words of a fresh context each time")
    for e in (s, c, t, x):
        e.close()
