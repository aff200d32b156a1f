"""Shapes of the seeded (compressed) key path and the reference side of its tests (test_seeded_shapes_premise.py on the CPU,
test_gpu_seeded.py on the GPU).

seeded_expand_kernel (csrc/seeded.cu) writes row g of a key as [mask_len stream words | body_len body words], 512 stream words per CTA:
  KSK: n_rows = k N l_ks LWE rows, mask_len = n,     body_len = 1
  BSK: n_rows = n_ggsw l (k + 1) GLWE rows, mask_len = k N, body_len = N   (n_ggsw = n, or (n / g) 2^g for multi-bit)
One set is kept per distinct (BSK shape, KSK shape, kernel family): the row lengths, row counts and the key layouts finish_bsk builds
are what change between them.  Keys are not encryptions: the bodies are uniform random words."""
import ctypes as C
from types import SimpleNamespace

import numpy as np

from fhe_string_bounty_b200 import _native as N

WORDS_PER_CTA = 512


def oracle_params(orc, name):
    """orc.Params of any classic ("<m>_<c>") or multi-bit ("multibit_<m>_<c>_g<g>") set from the engine's tables; the noise fields stay 0"""
    q = N.multi_bit_params(name[len("multibit_"):]) if name.startswith("multibit_") else N.classic_params(name)
    p = orc.Params()
    for k, v in q.items():
        setattr(p, k, v)
    return p


def kernel_family(q):
    """which PBS kernels a context of these parameters runs (c_api.cu tfhe_b200_ctx_create)"""
    n_, k, l, B, g = q["poly_size"], q["glwe_dim"], q["pbs_level"], q["pbs_base_log"], q["grouping_factor"]
    if n_ == 2048 and k == 1 and l == 1 and g != 2:
        return "multibit_v4_v8" if g == 3 else "classic_v4_v8"
    if n_ == 512 and k == 3 and l == 1 and g == 0:
        return "n512"
    if n_ == 8192 and k == 1 and l == 2 and 2 * B <= 31 and g == 0:
        return "n8192"
    if n_ >= 16384:
        return f"generic_big{n_.bit_length() - 1}"
    return "generic"


def all_sets():
    """the 36 classic and 6 multi-bit parameter sets (oracle.OTHER_MULTI_BIT_SETS plus multibit_2_2_g3) -> engine parameters"""
    out = {name: N.classic_params(name) for name in N._CLASSIC_SETS}
    for name in N._MULTI_BIT_SETS:
        out["multibit_" + name] = N.multi_bit_params(name)
    return out


def shape_key(q):
    bsk = (q["lwe_dim"], q["glwe_dim"], q["poly_size"], q["pbs_level"], q["grouping_factor"])
    ksk = (q["glwe_dim"] * q["poly_size"], q["lwe_dim"], q["ks_level"])
    return bsk, ksk, kernel_family(q)


def distinct_shapes():
    """shape key -> the first set that has it"""
    out = {}
    for name, q in all_sets().items():
        out.setdefault(shape_key(q), name)
    return out


SHAPES = list(distinct_shapes().values())
# every shape up to N = 8192 and one 3-level set each at N = 16384 and 32768 get full word equality against a standard upload of the
# reference key; the other N >= 16384 sets are checked on probe rows
FULL_BIG = ("1_6", "1_7")


def full_check(p, name):
    return p.poly_size <= 8192 or name in FULL_BIG


def ksk_stream(p):
    """(n_rows, mask_len, body_len) of the KSK as upload_seeded computes them"""
    return p.glwe_dim * p.poly_size * p.ks_level, p.lwe_dim, 1


def bsk_stream(p):
    """(n_rows, mask_len, body_len) of the BSK as upload_seeded computes them (bsk_poly_count / (k + 1) GLWE rows)"""
    k1 = p.glwe_dim + 1
    n_ggsw = (p.lwe_dim // p.grouping_factor) << p.grouping_factor if p.grouping_factor else p.lwe_dim
    return n_ggsw * p.pbs_level * k1, p.glwe_dim * p.poly_size, p.poly_size


def probe_rows(n_rows, mask_len):
    """rows of a stream worth reading back: 0; the first row whose mask crosses a 512-word CTA boundary; the row whose first word sits
    latest in its CTA and the row whose last word sits earliest in its CTA (the boundary one word into the mask, or one word before
    its end, when the lengths allow it); the first row after 0 that starts a CTA; the row that holds the first word of the last CTA;
    the last row (it holds the last word of the stream)"""
    r = np.arange(n_rows, dtype=np.int64)
    first, last = r * mask_len, (r + 1) * mask_len - 1
    rows = {0, n_rows - 1, int(np.argmax(first % WORDS_PER_CTA)), int(np.argmin(last % WORDS_PER_CTA))}
    for hit in (first // WORDS_PER_CTA != last // WORDS_PER_CTA, (first % WORDS_PER_CTA == 0) & (r > 0)):
        at = np.flatnonzero(hit)
        if at.size:
            rows.add(int(at[0]))
    grid = (n_rows * mask_len + WORDS_PER_CTA - 1) // WORDS_PER_CTA
    rows.add((WORDS_PER_CTA * (grid - 1)) // mask_len)
    return sorted(rows)


def stream_rows(orc, seed16, rows, mask_len):
    """mask words of the given rows straight from the AES-CTR stream: [len(rows), mask_len]"""
    out = np.zeros((len(rows), mask_len), dtype=np.uint64)
    for i, r in enumerate(rows):
        orc.lib().orc_csprng_mask_words(seed16, int(r) * mask_len, out[i], mask_len)
    return out


SEEDS = {
    "varied": bytes(range(0x11, 0x11 + 16)),
    "zeros": b"\x00" * 16,
    "ones": b"\xff" * 16,
}


def seed16(kind):
    return np.frombuffer(SEEDS[kind], dtype=np.uint8).copy()


class SeededKey:
    """A seeded KSK and BSK of one parameter set: 16 seed bytes each and uniform random bodies (light stand-in for
    oracle.CompressedServerKey: oracle/wire.py reads p, the seeds and the bodies)"""

    def __init__(self, orc, p, ksk_seed, bsk_seed, body_seed):
        L = orc.lib()
        self.orc, self.p = orc, p
        self.ksk_seed, self.bsk_seed = ksk_seed, bsk_seed
        rng = np.random.default_rng(body_seed)
        self.ksk_bodies = rng.integers(0, 2**64, size=L.orc_seeded_ksk_len(C.byref(p)), dtype=np.uint64)
        self.bsk_bodies = rng.integers(0, 2**64, size=L.orc_seeded_bsk_len(C.byref(p)), dtype=np.uint64)

    def ksk(self):
        """orc_decompress_seeded_ksk: the reference key in ServerKey's layout"""
        L = self.orc.lib()
        out = np.empty(L.orc_ksk_len(C.byref(self.p)), dtype=np.uint64)
        L.orc_decompress_seeded_ksk(C.byref(self.p), self.ksk_seed, self.ksk_bodies, out)
        return out

    def bsk(self):
        L = self.orc.lib()
        out = np.empty(L.orc_bsk_len(C.byref(self.p)), dtype=np.uint64)
        L.orc_decompress_seeded_bsk(C.byref(self.p), self.bsk_seed, self.bsk_bodies, out)
        return out

    def bsk_rows(self, rows):
        """GLWE rows of the reference BSK, [len(rows), (k + 1) N], from the stream and the bodies"""
        n_rows, mask_len, body_len = bsk_stream(self.p)
        return np.concatenate([stream_rows(self.orc, self.bsk_seed, rows, mask_len),
                               self.bsk_bodies.reshape(n_rows, body_len)[rows]], axis=1)

    def blob(self):
        from oracle import wire as W
        return W.serialize_compressed_server_key(self)


def seeded_key(orc, name, variant=0):
    """the key of a set: the seed pair rotates over varied bytes, all 0x00 and all 0xFF with the set's index"""
    p = oracle_params(orc, name)
    i = list(all_sets()).index(name) + variant
    kinds = list(SEEDS)
    return SeededKey(orc, p, seed16(kinds[i % 3]), seed16(kinds[(i + 1) % 3]), body_seed=0x5EED00 + 97 * i)


def mutated_params(orc, p, field):
    """p with one field changed to another value the wire parser accepts (its body counts follow the new dimensions; dimensions shrink
    where they can, to keep the blob small)"""
    r = orc.Params()
    for k, _ in orc.Params._fields_:
        setattr(r, k, getattr(p, k))
    v = getattr(p, field)
    if field == "grouping_factor":
        r.grouping_factor = 0 if v else 1
    elif field == "lwe_dim":
        r.lwe_dim = v - (p.grouping_factor or 1)
    elif field == "poly_size":
        r.poly_size = v // 2
    elif field in ("msg_mod", "carry_mod"):
        setattr(r, field, v * 2)
    else:
        setattr(r, field, v - 1 if v > 1 and field in ("glwe_dim", "pbs_level", "ks_level") else v + 1)
    return r


PARAM_FIELDS = ("lwe_dim", "glwe_dim", "poly_size", "pbs_base_log", "pbs_level", "ks_base_log", "ks_level", "grouping_factor",
                "msg_mod", "carry_mod")


def zero_body_key(orc, p):
    """a seeded key of parameters p with zero bodies (only its wire layout matters)"""
    L = orc.lib()
    return SimpleNamespace(p=p, ksk_seed=seed16("varied"), bsk_seed=seed16("varied"),
                           ksk_bodies=np.zeros(L.orc_seeded_ksk_len(C.byref(p)), dtype=np.uint64),
                           bsk_bodies=np.zeros(L.orc_seeded_bsk_len(C.byref(p)), dtype=np.uint64))
