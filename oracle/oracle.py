"""ctypes binding of the CPU oracle (oracle/tfhe_oracle.c).

TEST INFRASTRUCTURE ONLY -- see the header of oracle/tfhe_oracle.h.  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this module.
The product package (fhe_string_bounty_b200) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_SO = _HERE / "libtfhe_oracle.so"


def build(force: bool = False) -> Path:
    """Compile the C restatement (gcc -O3 -fopenmp).  Building the checker is not using it."""
    src = _HERE / "tfhe_oracle.c"
    hdr = _HERE / "tfhe_oracle.h"
    if force or not _SO.exists() or _SO.stat().st_mtime < max(src.stat().st_mtime, hdr.stat().st_mtime):
        subprocess.run(["make", "-C", str(_HERE), "-s", "-B"], check=True)
    return _SO


class Params(C.Structure):
    _fields_ = [
        ("lwe_dim", C.c_uint32), ("glwe_dim", C.c_uint32), ("poly_size", C.c_uint32),
        ("pbs_base_log", C.c_uint32), ("pbs_level", C.c_uint32),
        ("ks_base_log", C.c_uint32), ("ks_level", C.c_uint32),
        ("grouping_factor", C.c_uint32), ("msg_mod", C.c_uint32), ("carry_mod", C.c_uint32),
        ("lwe_std", C.c_double), ("glwe_std", C.c_double),
    ]

    @property
    def big_dim(self) -> int:
        return self.glwe_dim * self.poly_size

    @property
    def lut_len(self) -> int:
        return (self.glwe_dim + 1) * self.poly_size


class Rng(C.Structure):
    _fields_ = [("s", C.c_uint64 * 4), ("has_spare", C.c_int), ("spare", C.c_double)]


_lib = None
_u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")
_i64p = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
_u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
_PP = C.POINTER(Params)
_RP = C.POINTER(Rng)


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(str(_SO))
    sig = {
        "orc_params_message_2_carry_2_ks_pbs": (None, [_PP]),
        "orc_params_multi_bit_message_2_carry_2_group_3_ks_pbs": (None, [_PP]),
        "orc_params_toy": (None, [_PP]),
        "orc_rng_seed": (None, [_RP, C.c_uint64]),
        "orc_rng_u64": (C.c_uint64, [_RP]),
        "orc_gen_binary_key": (None, [_RP, _u64p, C.c_size_t]),
        "orc_lwe_encrypt": (None, [_u64p, C.c_size_t, C.c_uint64, C.c_double, _RP, _u64p]),
        "orc_lwe_decrypt": (C.c_uint64, [_u64p, C.c_size_t, _u64p]),
        "orc_gen_ksk": (None, [_PP, _u64p, _u64p, C.c_uint64, _u64p]),
        "orc_gen_bsk": (None, [_PP, _u64p, _u64p, C.c_uint64, _u64p]),
        "orc_gen_multi_bit_bsk": (None, [_PP, _u64p, _u64p, C.c_uint64, _u64p]),
        "orc_ksk_len": (C.c_size_t, [_PP]),
        "orc_bsk_len": (C.c_size_t, [_PP]),
        "orc_closest_representable": (C.c_uint64, [C.c_uint64, C.c_uint32, C.c_uint32]),
        "orc_closest_representable_u32": (C.c_uint32, [C.c_uint32, C.c_uint32, C.c_uint32]),
        "orc_decompose": (None, [C.c_uint64, C.c_uint32, C.c_uint32, _i64p]),
        "orc_modulus_switch": (C.c_uint64, [C.c_uint64, C.c_uint32]),
        "orc_monomial_div": (None, [_u64p, _u64p, C.c_size_t, C.c_size_t]),
        "orc_monomial_mul": (None, [_u64p, _u64p, C.c_size_t, C.c_size_t]),
        "orc_monomial_mul_and_subtract": (None, [_u64p, _u64p, C.c_size_t, C.c_size_t]),
        "orc_sample_extract0": (None, [_PP, _u64p, _u64p]),
        "orc_keyswitch": (None, [_PP, _u64p, _u64p, _u64p]),
        "orc_fill_accumulator": (C.c_uint64, [_PP, _u64p, _u64p]),
        "orc_trivial_pbs": (C.c_uint64, [_PP, C.c_uint64, _u64p]),
        "orc_encode": (C.c_uint64, [_PP, C.c_uint64]),
        "orc_decode": (C.c_uint64, [_PP, C.c_uint64]),
        "orc_fft_forward_integer": (None, [C.c_size_t, _u64p, _f64p, _f64p]),
        "orc_fft_forward_torus": (None, [C.c_size_t, _u64p, _f64p, _f64p]),
        "orc_fft_add_backward_torus": (None, [C.c_size_t, _u64p, _f64p, _f64p]),
        "orc_fourier_bsk_new": (C.c_void_p, [_PP, _u64p]),
        "orc_fourier_bsk_free": (None, [C.c_void_p]),
        "orc_add_external_product_f64": (None, [_PP, C.c_void_p, C.c_size_t, _u64p, _u64p]),
        "orc_add_external_product_exact": (None, [_PP, _u64p, _u64p, _u64p]),
        "orc_pbs_f64": (None, [_PP, C.c_void_p, _u64p, _u64p, _u64p]),
        "orc_pbs_f64_pow2_modulus": (None, [_PP, C.c_void_p, _u64p, _u64p, _u64p, C.c_uint32]),
        "orc_pbs_f64_partial": (None, [_PP, C.c_void_p, _u64p, _u64p, _u64p, C.c_size_t]),
        "orc_pbs_exact": (None, [_PP, _u64p, _u64p, _u64p, _u64p]),
        "orc_pbs_exact_steps": (None, [_PP, _u64p, _u64p, _u64p, _u64p, C.c_size_t]),
        "orc_pbs_exact_batch": (C.c_int, [_PP, _u64p, _u64p, C.c_void_p, _u64p, _u64p, C.c_size_t, C.c_size_t, C.c_int]),
        "orc_pbs_f64_batch": (C.c_int, [_PP, C.c_void_p, _u64p, C.c_void_p, _u64p, _u64p, C.c_size_t, C.c_size_t, C.c_int]),
        "orc_ks_pbs_batch": (C.c_int, [_PP, _u64p, C.c_void_p, _u64p, C.c_void_p, _u64p, _u64p, C.c_void_p, C.c_size_t, C.c_int]),
        "orc_max_threads": (C.c_int, []),
        "orc_aes_sbox": (C.POINTER(C.c_uint8), []),
        "orc_aes128_expand_key": (None, [_u8p, _u8p]),
        "orc_aes128_encrypt_block": (None, [_u8p, _u8p, _u8p]),
        "orc_csprng_table_bytes": (None, [_u8p, C.c_uint64, _u8p, C.c_size_t]),
        "orc_csprng_generate_bytes": (None, [_u8p, C.c_uint64, _u8p, C.c_size_t]),
        "orc_csprng_mask_words": (None, [_u8p, C.c_uint64, _u64p, C.c_size_t]),
        "orc_seeded_bsk_len": (C.c_size_t, [_PP]),
        "orc_seeded_ksk_len": (C.c_size_t, [_PP]),
        "orc_decompress_seeded_bsk": (None, [_PP, _u8p, _u64p, _u64p]),
        "orc_decompress_seeded_ksk": (None, [_PP, _u8p, _u64p, _u64p]),
        "orc_compress_bsk": (None, [_PP, _u64p, _u8p, _u64p, _u64p]),
        "orc_compress_ksk": (None, [_PP, _u64p, _u8p, _u64p, _u64p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def params(name: str = "2_2") -> Params:
    p = Params()
    L = lib()
    if name in ("2_2", "PARAM_MESSAGE_2_CARRY_2_KS_PBS"):
        L.orc_params_message_2_carry_2_ks_pbs(C.byref(p))
    elif name in ("multibit_2_2_g3", "PARAM_MULTI_BIT_MESSAGE_2_CARRY_2_GROUP_3_KS_PBS"):
        L.orc_params_multi_bit_message_2_carry_2_group_3_ks_pbs(C.byref(p))
    elif name == "toy":
        L.orc_params_toy(C.byref(p))
    elif name in OTHER_CLASSIC_SETS:
        (p.lwe_dim, p.glwe_dim, p.poly_size, p.lwe_std, p.glwe_std, p.pbs_base_log, p.pbs_level, p.ks_level, p.ks_base_log,
         p.msg_mod, p.carry_mod) = OTHER_CLASSIC_SETS[name]
        p.grouping_factor = 0
    elif name in OTHER_MULTI_BIT_SETS:
        (p.lwe_dim, p.glwe_dim, p.poly_size, p.lwe_std, p.glwe_std, p.pbs_base_log, p.pbs_level, p.ks_base_log, p.ks_level,
         p.msg_mod, p.carry_mod, p.grouping_factor) = OTHER_MULTI_BIT_SETS[name]
    else:
        raise KeyError(name)
    return p


# PARAM_MULTI_BIT_MESSAGE_<m>_CARRY_<c>_GROUP_<g>_KS_PBS, name "multibit_<m>_<c>_g<g>" (shortint/parameters/multi_bit.rs), fields:
# lwe_dimension, glwe_dimension, polynomial_size, lwe_modular_std_dev, glwe_modular_std_dev, pbs_base_log, pbs_level, ks_base_log,
# ks_level, message_modulus, carry_modulus, grouping_factor
OTHER_MULTI_BIT_SETS = {
    "multibit_1_1_g2": (764, 3, 512, 0.000006025673585415336, 0.0000000000039666089171633006, 18, 1, 6, 2, 2, 2, 2),          # :96
    "multibit_2_2_g2": (818, 1, 2048, 0.000002226459789930014, 0.0000000000000003152931493498455, 22, 1, 5, 3, 4, 4, 2),        # :115
    "multibit_3_3_g2": (922, 1, 8192, 0.0000003272369292345697, 0.0000000000000000002168404344971009, 14, 2, 4, 4, 8, 8, 2),    # :134
    "multibit_1_1_g3": (765, 3, 512, 0.000005915594083804978, 0.0000000000039666089171633006, 18, 1, 6, 2, 2, 2, 3),           # :154
    "multibit_3_3_g3": (972, 1, 8192, 0.00000013016688349592805, 0.0000000000000000002168404344971009, 14, 2, 6, 3, 8, 8, 3),   # :192
}


# PARAM_MESSAGE_<m>_CARRY_<c>_KS_PBS, name "<m>_<c>" (shortint/parameters/mod.rs:598-911), fields in the order of the struct literal:
# lwe_dimension, glwe_dimension, polynomial_size, lwe_modular_std_dev, glwe_modular_std_dev, pbs_base_log, pbs_level, ks_level,
# ks_base_log, message_modulus, carry_modulus
OTHER_CLASSIC_SETS = {
    "1_0": (678, 5, 256, 0.000022810107419132102, 0.00000000037411618952047216, 15, 1, 2, 5, 2, 1),  # :598-612
    "1_1": (684, 3, 512, 0.00002043784477291318, 0.0000000000034525330484572114, 18, 1, 3, 4, 2, 2),  # :613-627
    "2_0": (656, 2, 512, 0.000034119201269311964, 0.00000004053919869756513, 8, 2, 4, 3, 4, 1),  # :628-642
    "1_2": (742, 2, 1024, 0.000007069849454709433, 0.00000000000000029403601535432533, 23, 1, 3, 4, 2, 4),  # :643-657
    "1_3": (745, 1, 2048, 0.000006692125069956277, 0.00000000000000029403601535432533, 23, 1, 5, 3, 2, 8),  # :688-702
    "1_4": (807, 1, 4096, 0.0000021515145918907506, 0.0000000000000000002168404344971009, 15, 2, 5, 3, 2, 16),  # :748-762
    "2_3": (856, 1, 4096, 0.0000008775214009854235, 0.0000000000000000002168404344971009, 22, 1, 6, 3, 4, 8),  # :763-777
    "3_3": (864, 1, 8192, 0.000000757998020150446, 0.0000000000000000002168404344971009, 15, 2, 6, 3, 8, 8),  # :853-867
    "4_3": (930, 1, 16384, 0.00000022649232786295453, 0.0000000000000000002168404344971009, 15, 2, 6, 3, 16, 8),  # :958-972
    "4_4": (996, 1, 32768, 0.00000006767666038309478, 0.0000000000000000002168404344971009, 15, 2, 7, 3, 16, 16),  # :1063-1077
}


class ClientKey:
    """Secret keys of shortint::ClientKey (engine/client_side.rs:13-37): GLWE key, its flattened
    'big' LWE view, and the small LWE key.  encrypt/decrypt follow client_side.rs:58-124 and
    client_key/mod.rs:281-302 (Big encryption key => ciphertexts under the big key, GLWE noise)."""

    def __init__(self, p: Params, seed: int):
        L = lib()
        self.p = p
        self.rng = Rng()
        L.orc_rng_seed(C.byref(self.rng), seed)
        self.glwe_sk = np.zeros(p.big_dim, dtype=np.uint64)
        self.small_sk = np.zeros(p.lwe_dim, dtype=np.uint64)
        L.orc_gen_binary_key(C.byref(self.rng), self.glwe_sk, p.big_dim)
        L.orc_gen_binary_key(C.byref(self.rng), self.small_sk, p.lwe_dim)
        self.big_sk = self.glwe_sk  # GlweSecretKey::as_lwe_secret_key

    def encrypt_raw(self, plaintext: int) -> np.ndarray:
        ct = np.zeros(self.p.big_dim + 1, dtype=np.uint64)
        lib().orc_lwe_encrypt(self.big_sk, self.p.big_dim, plaintext & (2**64 - 1), self.p.glwe_std, C.byref(self.rng), ct)
        return ct

    def encrypt(self, msg: int) -> np.ndarray:
        """client_side.rs:58-85: message reduced mod msg_mod*carry_mod? No: mod message modulus."""
        m = msg % self.p.msg_mod
        return self.encrypt_raw(lib().orc_encode(C.byref(self.p), m))

    def encrypt_with_carry(self, value: int) -> np.ndarray:
        """Encrypt any value below msg_mod*carry_mod (used to exercise every LUT box)."""
        v = value % (self.p.msg_mod * self.p.carry_mod)
        return self.encrypt_raw(lib().orc_encode(C.byref(self.p), v))

    def encrypt_batch(self, values) -> np.ndarray:
        return np.stack([self.encrypt_with_carry(int(v)) for v in values])

    def decrypt_raw(self, ct: np.ndarray) -> int:
        return int(lib().orc_lwe_decrypt(self.big_sk, self.p.big_dim, np.ascontiguousarray(ct)))

    def decrypt_message_and_carry(self, ct: np.ndarray) -> int:
        return int(lib().orc_decode(C.byref(self.p), self.decrypt_raw(ct)))

    def decrypt(self, ct: np.ndarray) -> int:
        return self.decrypt_message_and_carry(ct) % self.p.msg_mod

    def decrypt_batch(self, cts: np.ndarray) -> np.ndarray:
        return np.array([self.decrypt_message_and_carry(c) for c in cts], dtype=np.int64)

    def decrypt_small_raw(self, ct: np.ndarray) -> int:
        return int(lib().orc_lwe_decrypt(self.small_sk, self.p.lwe_dim, np.ascontiguousarray(ct)))


class ServerKey:
    """KSK + (multi-bit) BSK in the standard domain, plus the oracle's own Fourier copy
    (shortint/engine/server_side.rs:54-160)."""

    def __init__(self, ck: ClientKey, seed: int, fourier: bool = True):
        L = lib()
        p = ck.p
        self.p = p
        self.ksk = np.zeros(L.orc_ksk_len(C.byref(p)), dtype=np.uint64)
        L.orc_gen_ksk(C.byref(p), ck.big_sk, ck.small_sk, seed, self.ksk)
        self.bsk = np.zeros(L.orc_bsk_len(C.byref(p)), dtype=np.uint64)
        if p.grouping_factor == 0:
            L.orc_gen_bsk(C.byref(p), ck.small_sk, ck.glwe_sk, seed + 1, self.bsk)
        else:
            L.orc_gen_multi_bit_bsk(C.byref(p), ck.small_sk, ck.glwe_sk, seed + 1, self.bsk)
        self._fourier = None
        if fourier:
            self._fourier = L.orc_fourier_bsk_new(C.byref(p), self.bsk)

    def __del__(self):
        if getattr(self, "_fourier", None):
            lib().orc_fourier_bsk_free(self._fourier)
            self._fourier = None

    @property
    def fourier(self):
        if self._fourier is None:
            self._fourier = lib().orc_fourier_bsk_new(C.byref(self.p), self.bsk)
        return self._fourier

    # shortint/server_key/mod.rs:383-399
    def generate_lookup_table(self, f) -> tuple[np.ndarray, int]:
        p = self.p
        table = np.array([int(f(i)) for i in range(p.msg_mod * p.carry_mod)], dtype=np.uint64)
        acc = np.zeros(p.lut_len, dtype=np.uint64)
        degree = lib().orc_fill_accumulator(C.byref(p), table, acc)
        return acc, int(degree)

    # shortint/server_key/bivariate_pbs.rs:71-97
    def generate_lookup_table_bivariate(self, f) -> tuple[np.ndarray, int]:
        m = self.p.msg_mod
        return self.generate_lookup_table(lambda x: f((x // m) % m, (x % m) % m))

    def keyswitch(self, ct: np.ndarray) -> np.ndarray:
        out = np.zeros(self.p.lwe_dim + 1, dtype=np.uint64)
        lib().orc_keyswitch(C.byref(self.p), self.ksk, np.ascontiguousarray(ct), out)
        return out

    def pbs(self, lwe_small: np.ndarray, acc: np.ndarray, exact: bool = False) -> np.ndarray:
        out = np.zeros(self.p.big_dim + 1, dtype=np.uint64)
        if exact:
            lib().orc_pbs_exact(C.byref(self.p), self.bsk, np.ascontiguousarray(lwe_small), acc, out)
        else:
            lib().orc_pbs_f64(C.byref(self.p), self.fourier, np.ascontiguousarray(lwe_small), acc, out)
        return out

    def pbs_partial(self, lwe_small: np.ndarray, acc: np.ndarray, n_steps: int) -> np.ndarray:
        """PBS stopped after n_steps mask elements (classic) / groups (multi-bit): what tfhe_b200_pbs_batch_partial computes."""
        out = np.zeros(self.p.big_dim + 1, dtype=np.uint64)
        lib().orc_pbs_f64_partial(C.byref(self.p), self.fourier, np.ascontiguousarray(lwe_small), np.ascontiguousarray(acc), out, n_steps)
        return out

    def pbs_pow2_modulus(self, lwe_small: np.ndarray, acc: np.ndarray, log2_q: int) -> np.ndarray:
        """PBS under a non-native power-of-two ciphertext modulus 2^log2_q (bootstrap.rs:318-330)."""
        out = np.zeros(self.p.big_dim + 1, dtype=np.uint64)
        lib().orc_pbs_f64_pow2_modulus(C.byref(self.p), self.fourier, np.ascontiguousarray(lwe_small), acc, out, log2_q)
        return out

    def ks_pbs_batch(self, cts: np.ndarray, luts: np.ndarray, lut_idx=None, threads: int = 0, want_ks: bool = False):
        """shortint/server_key/mod.rs:783-857 over a batch (one ciphertext per OpenMP thread)."""
        p = self.p
        cts = np.ascontiguousarray(cts, dtype=np.uint64).reshape(-1, p.big_dim + 1)
        luts = np.ascontiguousarray(luts, dtype=np.uint64).reshape(-1, p.lut_len)
        batch = cts.shape[0]
        out = np.zeros_like(cts)
        idx_ptr = None
        if lut_idx is not None:
            lut_idx = np.ascontiguousarray(lut_idx, dtype=np.uint32)
            idx_ptr = lut_idx.ctypes.data_as(C.c_void_p)
        ks = np.zeros((batch, p.lwe_dim + 1), dtype=np.uint64) if want_ks else None
        ks_ptr = ks.ctypes.data_as(C.c_void_p) if want_ks else None
        used = lib().orc_ks_pbs_batch(C.byref(p), self.ksk, self.fourier, luts, idx_ptr, cts, out, ks_ptr, batch, threads)
        self.last_threads = used
        return (out, ks) if want_ks else out


class FourierKey:
    """The oracle's Fourier copy of an explicit standard-domain (multi-bit) BSK, e.g. a test key that is not an encryption."""

    def __init__(self, p: Params, bsk: np.ndarray):
        self.p = p
        self.ptr = lib().orc_fourier_bsk_new(C.byref(p), np.ascontiguousarray(bsk, dtype=np.uint64))

    def __del__(self):
        if getattr(self, "ptr", None):
            lib().orc_fourier_bsk_free(self.ptr)
            self.ptr = None


def _pbs_batch(fn, p: Params, key, small, luts, lut_idx, max_steps, threads):
    small = np.ascontiguousarray(small, dtype=np.uint64).reshape(-1, p.lwe_dim + 1)
    luts = np.ascontiguousarray(luts, dtype=np.uint64).reshape(-1, p.lut_len)
    out = np.zeros((small.shape[0], p.big_dim + 1), dtype=np.uint64)
    idx_ptr = None
    if lut_idx is not None:
        lut_idx = np.ascontiguousarray(lut_idx, dtype=np.uint32)
        assert lut_idx.shape == (small.shape[0],) and (small.shape[0] == 0 or int(lut_idx.max()) < luts.shape[0])
        idx_ptr = lut_idx.ctypes.data_as(C.c_void_p)
    steps = C.c_size_t(-1).value if max_steps is None else int(max_steps)
    fn(C.byref(p), key, luts, idx_ptr, small, out, small.shape[0], steps, threads)
    return out


def pbs_exact_batch(p: Params, bsk: np.ndarray, small, luts, lut_idx=None, max_steps=None, threads: int = 0) -> np.ndarray:
    """Exact integer PBS (classic or multi-bit) of a batch under an explicit standard-domain BSK, stopped after max_steps mask elements /
    groups (None: the whole rotation).  Cost O(n * (k+1)^2 * l * N * nnz) per ciphertext, nnz = nonzeros per key polynomial."""
    bsk = np.ascontiguousarray(bsk, dtype=np.uint64)
    assert bsk.size == lib().orc_bsk_len(C.byref(p))
    return _pbs_batch(lib().orc_pbs_exact_batch, p, bsk, small, luts, lut_idx, max_steps, threads)


def pbs_f64_batch(p: Params, fourier: FourierKey, small, luts, lut_idx=None, max_steps=None, threads: int = 0) -> np.ndarray:
    """The oracle's f64 PBS (what orc_pbs_f64_partial computes) over a batch, same arguments as pbs_exact_batch."""
    return _pbs_batch(lib().orc_pbs_f64_batch, p, fourier.ptr, small, luts, lut_idx, max_steps, threads)


def decompose(x: int, base_log: int, level: int) -> list[int]:
    d = np.zeros(level, dtype=np.int64)
    lib().orc_decompose(x, base_log, level, d)
    return [int(v) for v in d]


def seed_bytes(seed: int) -> np.ndarray:
    """concrete-csprng Seed(u128) -> the 16 key bytes the block cipher sees (soft/block_cipher.rs:16: to_ne_bytes, little endian)."""
    return np.frombuffer(int(seed).to_bytes(16, "little"), dtype=np.uint8).copy()


class CompressedServerKey:
    """shortint::CompressedServerKey (shortint/server_key/mod.rs:935-1023): seeded KSK + seeded (multi-bit) BSK, i.e. one compression
    seed per key plus the ciphertext bodies.  Built here from a ServerKey by re-drawing every mask from the seeded stream (test-side
    key generation); decompress() restates seeded_lwe_keyswitch_key_decompression.rs / seeded_lwe_bootstrap_key_decompression.rs."""

    def __init__(self, ck: ClientKey, sk: ServerKey, ksk_seed: int, bsk_seed: int):
        L = lib()
        p = sk.p
        self.p = p
        self.ksk_seed, self.bsk_seed = seed_bytes(ksk_seed), seed_bytes(bsk_seed)
        self.ksk_bodies = np.zeros(L.orc_seeded_ksk_len(C.byref(p)), dtype=np.uint64)
        self.bsk_bodies = np.zeros(L.orc_seeded_bsk_len(C.byref(p)), dtype=np.uint64)
        L.orc_compress_ksk(C.byref(p), ck.small_sk, self.ksk_seed, sk.ksk, self.ksk_bodies)
        L.orc_compress_bsk(C.byref(p), ck.glwe_sk, self.bsk_seed, sk.bsk, self.bsk_bodies)

    def decompress(self):
        """-> (ksk, bsk) in the standard layouts of ServerKey"""
        L = lib()
        p = self.p
        ksk = np.zeros(L.orc_ksk_len(C.byref(p)), dtype=np.uint64)
        bsk = np.zeros(L.orc_bsk_len(C.byref(p)), dtype=np.uint64)
        L.orc_decompress_seeded_ksk(C.byref(p), self.ksk_seed, self.ksk_bodies, ksk)
        L.orc_decompress_seeded_bsk(C.byref(p), self.bsk_seed, self.bsk_bodies, bsk)
        return ksk, bsk
