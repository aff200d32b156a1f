"""ctypes loader for libtfhe_b200.so and a small numpy-facing wrapper around the C ABI.

Nothing here computes: every method forwards to an ``extern "C"`` entry point declared in
``include/tfhe_b200.h`` (EXPORTS), ``include/tfhe_b200_sharded.h`` (SHARDED_EXPORTS) or ``include/tfhe_b200_many_lut.h``
(MANY_LUT_EXPORTS).  Missing library or missing GPU
raises NativeError (no fallback).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_PKG = Path(__file__).resolve().parent
_SO = _PKG / "libtfhe_b200.so"
_SOURCES = ["csrc/pbs_v4.cu", "csrc/pbs_v8.cu", "csrc/pbs_multibit_v4.cu", "csrc/pbs_multibit_v8.cu", "csrc/pbs_generic.cu", "csrc/pbs_n512.cu", "csrc/pbs_n8192.cu", "csrc/keyswitch.cu", "csrc/keyswitch_mma.cu", "csrc/keyswitch_tc.cu", "csrc/leveled.cu", "csrc/seeded.cu", "csrc/probe.cu", "csrc/exchange.cu", "csrc/c_api.cu", "csrc/host_api.cu"]
_HEADERS = ["csrc/fft_core.cuh", "csrc/fft16_core.cuh", "csrc/fft8_core.cuh", "csrc/fft16x_slots.cuh", "csrc/pbs16_common.cuh", "csrc/pbs8_common.cuh", "csrc/ring_helpers.cuh", "csrc/sample_extract.cuh", "csrc/kernels.h", "csrc/ctx.h", "csrc/host/program.h", "csrc/host/radix.h", "csrc/host/strings.h", "csrc/host/padded.h", "../include/tfhe_b200.h", "../include/tfhe_b200_sharded.h", "../include/tfhe_b200_many_lut.h"]

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "-shared",
]


class NativeError(RuntimeError):
    pass


def build_native(force: bool = False, verbose: bool = False) -> Path:
    """nvcc-compile every kernel for sm_100a into the in-tree libtfhe_b200.so."""
    srcs = [_PKG / s for s in _SOURCES if (_PKG / s).exists()]
    deps = srcs + [(_PKG / h).resolve() for h in _HEADERS]
    if not force and _SO.exists() and all(_SO.stat().st_mtime >= d.stat().st_mtime for d in deps if d.exists()):
        return _SO
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    build_dir = _PKG / "build"
    build_dir.mkdir(exist_ok=True)
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"]

    def compile_one(src: Path):
        obj = build_dir / (src.stem + ".o")
        cmd = [nvcc, *compile_flags, "-c", "-o", str(obj), str(src)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        res = subprocess.run(cmd, capture_output=True, text=True, env=env)
        return obj, res

    # one nvcc per translation unit, in parallel (the kernels are independent), then one link step
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as pool:
        results = list(pool.map(compile_one, srcs))
    log = ""
    for obj, res in results:
        log += res.stderr
        if res.returncode != 0:
            raise NativeError("nvcc failed:\n" + res.stdout + res.stderr)
    res = subprocess.run([nvcc, "-shared", "-o", str(_SO), *[str(o) for o, _ in results]], capture_output=True, text=True, env=env)
    if res.returncode != 0:
        raise NativeError("nvcc link failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(log)
    return _SO


class Params(C.Structure):
    """Mirror of tfhe_b200_params (shortint ClassicPBSParameters subset)."""
    _fields_ = [
        ("lwe_dim", C.c_uint32), ("glwe_dim", C.c_uint32), ("poly_size", C.c_uint32),
        ("pbs_base_log", C.c_uint32), ("pbs_level", C.c_uint32),
        ("ks_base_log", C.c_uint32), ("ks_level", C.c_uint32),
        ("grouping_factor", C.c_uint32), ("msg_mod", C.c_uint32), ("carry_mod", C.c_uint32),
    ]

    @property
    def big_len(self) -> int:
        return self.glwe_dim * self.poly_size + 1

    @property
    def small_len(self) -> int:
        return self.lwe_dim + 1

    @property
    def lut_len(self) -> int:
        return (self.glwe_dim + 1) * self.poly_size

    @property
    def ksk_len(self) -> int:
        return self.glwe_dim * self.poly_size * self.ks_level * (self.lwe_dim + 1)

    @property
    def bsk_len(self) -> int:
        k1 = self.glwe_dim + 1
        n_ggsw = self.lwe_dim if not self.grouping_factor else (self.lwe_dim // self.grouping_factor) << self.grouping_factor
        return n_ggsw * self.pbs_level * k1 * k1 * self.poly_size


# shortint/parameters/mod.rs:703-717
PARAM_MESSAGE_2_CARRY_2_KS_PBS = dict(lwe_dim=742, glwe_dim=1, poly_size=2048, pbs_base_log=23, pbs_level=1,
                                      ks_base_log=3, ks_level=5, grouping_factor=0, msg_mod=4, carry_mod=4)

# shortint/parameters/multi_bit.rs:173-190
PARAM_MULTI_BIT_MESSAGE_2_CARRY_2_GROUP_3_KS_PBS = dict(lwe_dim=888, glwe_dim=1, poly_size=2048, pbs_base_log=21, pbs_level=1,
                                                        ks_base_log=7, ks_level=2, grouping_factor=3, msg_mod=4, carry_mod=4)

# every PARAM_MESSAGE_<m>_CARRY_<c>_KS_PBS of shortint/parameters/mod.rs:598-1136, keyed "<m>_<c>":
# (lwe_dim, glwe_dim, poly_size, pbs_base_log, pbs_level, ks_base_log, ks_level, msg_mod, carry_mod)
_CLASSIC_SETS = {
    "1_0": (678, 5, 256, 15, 1, 5, 2, 2, 1),  # :598
    "1_1": (684, 3, 512, 18, 1, 4, 3, 2, 2),  # :613
    "2_0": (656, 2, 512, 8, 2, 3, 4, 4, 1),  # :628
    "1_2": (742, 2, 1024, 23, 1, 4, 3, 2, 4),  # :643
    "2_1": (742, 2, 1024, 23, 1, 4, 3, 4, 2),  # :658
    "3_0": (742, 2, 1024, 23, 1, 4, 3, 8, 1),  # :673
    "1_3": (745, 1, 2048, 23, 1, 3, 5, 2, 8),  # :688
    "2_2": (742, 1, 2048, 23, 1, 3, 5, 4, 4),  # :703
    "3_1": (742, 1, 2048, 23, 1, 3, 5, 8, 2),  # :718
    "4_0": (742, 1, 2048, 23, 1, 3, 5, 16, 1),  # :733
    "1_4": (807, 1, 4096, 15, 2, 3, 5, 2, 16),  # :748
    "2_3": (856, 1, 4096, 22, 1, 3, 6, 4, 8),  # :763
    "3_2": (812, 1, 4096, 22, 1, 3, 5, 8, 4),  # :778
    "4_1": (808, 1, 4096, 22, 1, 3, 5, 16, 2),  # :793
    "5_0": (807, 1, 4096, 22, 1, 3, 5, 32, 1),  # :808
    "1_5": (864, 1, 8192, 15, 2, 3, 6, 2, 32),  # :823
    "2_4": (864, 1, 8192, 15, 2, 3, 6, 4, 16),  # :838
    "3_3": (864, 1, 8192, 15, 2, 3, 6, 8, 8),  # :853
    "4_2": (864, 1, 8192, 15, 2, 3, 6, 16, 4),  # :868
    "5_1": (875, 1, 8192, 22, 1, 3, 6, 32, 2),  # :883
    "6_0": (915, 1, 8192, 22, 1, 4, 4, 64, 1),  # :898
    "1_6": (930, 1, 16384, 11, 3, 3, 6, 2, 64),  # :913
    "2_5": (934, 1, 16384, 15, 2, 3, 6, 4, 32),  # :928
    "3_4": (930, 1, 16384, 15, 2, 3, 6, 8, 16),  # :943
    "4_3": (930, 1, 16384, 15, 2, 3, 6, 16, 8),  # :958
    "5_2": (930, 1, 16384, 15, 2, 3, 6, 32, 4),  # :973
    "6_1": (930, 1, 16384, 15, 2, 3, 6, 64, 2),  # :988
    "7_0": (930, 1, 16384, 15, 2, 3, 6, 128, 1),  # :1003
    "1_7": (1004, 1, 32768, 11, 3, 3, 7, 2, 128),  # :1018
    "2_6": (987, 1, 32768, 11, 3, 3, 7, 4, 64),  # :1033
    "3_5": (985, 1, 32768, 11, 3, 3, 7, 8, 32),  # :1048
    "4_4": (996, 1, 32768, 15, 2, 3, 7, 16, 16),  # :1063
    "5_3": (1020, 1, 32768, 15, 2, 4, 5, 32, 8),  # :1078
    "6_2": (1018, 1, 32768, 15, 2, 4, 5, 64, 4),  # :1093
    "7_1": (1017, 1, 32768, 15, 2, 4, 5, 128, 2),  # :1108
    "8_0": (1017, 1, 32768, 15, 2, 4, 5, 256, 1),  # :1123
}


def classic_params(name: str) -> dict:
    """PARAM_MESSAGE_<m>_CARRY_<c>_KS_PBS as the keyword arguments of Params; name = "<m>_<c>" (e.g. "2_2", "3_3", "4_4")."""
    t = _CLASSIC_SETS[name]
    return dict(lwe_dim=t[0], glwe_dim=t[1], poly_size=t[2], pbs_base_log=t[3], pbs_level=t[4], ks_base_log=t[5], ks_level=t[6],
                grouping_factor=0, msg_mod=t[7], carry_mod=t[8])

# every PARAM_MULTI_BIT_MESSAGE_<m>_CARRY_<c>_GROUP_<g>_KS_PBS of shortint/parameters/multi_bit.rs:96-209, keyed "<m>_<c>_g<g>":
# (lwe_dim, glwe_dim, poly_size, pbs_base_log, pbs_level, ks_base_log, ks_level, msg_mod, carry_mod, grouping_factor)
_MULTI_BIT_SETS = {
    "1_1_g2": (764, 3, 512, 18, 1, 6, 2, 2, 2, 2),   # :96
    "2_2_g2": (818, 1, 2048, 22, 1, 5, 3, 4, 4, 2),  # :115
    "3_3_g2": (922, 1, 8192, 14, 2, 4, 4, 8, 8, 2),  # :134
    "1_1_g3": (765, 3, 512, 18, 1, 6, 2, 2, 2, 3),   # :154
    "2_2_g3": (888, 1, 2048, 21, 1, 7, 2, 4, 4, 3),  # :173
    "3_3_g3": (972, 1, 8192, 14, 2, 6, 3, 8, 8, 3),  # :192
}


def multi_bit_params(name: str) -> dict:
    """PARAM_MULTI_BIT_MESSAGE_<m>_CARRY_<c>_GROUP_<g>_KS_PBS as the keyword arguments of Params; name = "<m>_<c>_g<g>"."""
    t = _MULTI_BIT_SETS[name]
    return dict(lwe_dim=t[0], glwe_dim=t[1], poly_size=t[2], pbs_base_log=t[3], pbs_level=t[4], ks_base_log=t[5], ks_level=t[6],
                msg_mod=t[7], carry_mod=t[8], grouping_factor=t[9])


EXPORTS = {
    "tfhe_b200_ctx_create": (C.c_int, [C.c_int, C.POINTER(Params), C.POINTER(C.c_void_p)]),
    "tfhe_b200_ctx_destroy": (C.c_int, [C.c_void_p]),
    "tfhe_b200_set_ciphertext_modulus_log2": (C.c_int, [C.c_void_p, C.c_uint32]),
    "tfhe_b200_last_error": (C.c_char_p, []),
    "tfhe_b200_upload_ksk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "tfhe_b200_upload_bsk_std": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "tfhe_b200_upload_seeded_ksk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tfhe_b200_upload_seeded_bsk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tfhe_b200_upload_luts": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32]),
    "tfhe_b200_wire_parse_compressed_server_key": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p]),
    "tfhe_b200_load_compressed_server_key": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "tfhe_b200_wire_read_ciphertexts": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                                                  C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "tfhe_b200_wire_write_ciphertexts": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_size_t,
                                                   C.POINTER(C.c_size_t)]),
    "tfhe_b200_keyswitch_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tfhe_b200_pbs_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tfhe_b200_ks_pbs_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tfhe_b200_pbs_ks_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tfhe_b200_keyswitch_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "tfhe_b200_pbs_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "tfhe_b200_ks_pbs_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "tfhe_b200_synchronize": (C.c_int, [C.c_void_p]),
    "tfhe_b200_pbs_batch_partial": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32]),
    "tfhe_b200_set_tuning": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "tfhe_b200_kernel_launches": (C.c_uint64, [C.c_void_p]),
    "tfhe_b200_time_last_kernels": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "tfhe_b200_probe_fp64_tflops": (C.c_int, [C.c_int, C.POINTER(C.c_double)]),
    "tfhe_b200_version": (C.c_char_p, []),
    "tfhe_b200_plan_classic_level": (None, [C.c_size_t, C.c_uint32, C.c_size_t, C.c_int, C.POINTER(C.c_size_t)]),
    "tfhe_b200_program_build": (C.c_int, [C.POINTER(Params), C.c_char_p, C.c_void_p, C.c_size_t, C.c_char_p, C.POINTER(C.c_void_p)]),
    "tfhe_b200_program_destroy": (C.c_int, [C.c_void_p]),
    "tfhe_b200_program_counts": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tfhe_b200_program_copy": (C.c_int, [C.c_void_p] + [C.c_void_p] * 11),
    "tfhe_b200_program_accumulators": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tfhe_b200_program_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tfhe_b200_program_run_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tfhe_b200_program_last_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "tfhe_b200_exchange_create": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]),
    "tfhe_b200_exchange_handle": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tfhe_b200_exchange_attach": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tfhe_b200_exchange_attach_local": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "tfhe_b200_exchange_send_rows": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "tfhe_b200_exchange_gather_stride": (C.c_size_t, [C.c_void_p, C.c_uint32]),
    "tfhe_b200_exchange_all_gather": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "tfhe_b200_exchange_all_reduce_sum": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "tfhe_b200_exchange_group_run": (C.c_int, [C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p), C.c_int, C.c_void_p]),
    "tfhe_b200_exchange_destroy": (C.c_int, [C.c_void_p]),
}

# include/tfhe_b200_sharded.h: any recorded program across the ranks of an exchange
SHARDED_EXPORTS = {
    "tfhe_b200_program_shard_plan": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p]),
    "tfhe_b200_program_level_share": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p]),
    "tfhe_b200_program_run_sharded": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "tfhe_b200_program_run_sharded_group": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_uint32,
                                                      C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_uint64, C.c_void_p]),
}

# include/tfhe_b200_many_lut.h: many-LUT PBS
MANY_LUT_EXPORTS = {
    "tfhe_b200_upload_many_luts": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "tfhe_b200_pbs_many_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tfhe_b200_pbs_many_batch_partial": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32]),
    "tfhe_b200_ks_pbs_many_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tfhe_b200_pbs_many_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "tfhe_b200_ks_pbs_many_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
}

_lib = None


def many_lut_accumulator(params: dict | Params, fns) -> np.ndarray:
    """tfhe-rs generate_many_lookup_table (shortint/server_key/mod.rs): the (k + 1) * N accumulator that stacks the F = len(fns)
    functions, f_f(x) * Delta in box f * chunk + x for x < chunk = total // F (total = msg_mod * carry_mod), 0 in the boxes from F * chunk
    on, then the half-box negation and rotation of generate_lookup_table.  Upload with Engine.upload_many_luts."""
    p = params if isinstance(params, Params) else Params(**params)
    total, N = p.msg_mod * p.carry_mod, p.poly_size
    F = len(fns)
    if not 2 <= F <= total:
        raise ValueError(f"a many-LUT accumulator holds 2 ... msg_mod * carry_mod = {total} functions, not {F}")
    chunk, box = total // F, N // total
    delta = (1 << 63) // total
    boxes = np.zeros(total, dtype=np.uint64)
    for f, fn in enumerate(fns):
        for x in range(chunk):
            boxes[f * chunk + x] = (int(fn(x)) * delta) & (2**64 - 1)
    body = np.repeat(boxes, box)
    half = box // 2
    body[:half] = np.uint64(0) - body[:half]
    acc = np.zeros(p.lut_len, dtype=np.uint64)
    acc[p.glwe_dim * N:] = np.roll(body, -half)
    return acc


def load_native():
    """dlopen the in-tree library and type every exported symbol; raises NativeError if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not _SO.exists():
        raise NativeError(f"{_SO} is missing: run __graft_entry__.build() (nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(str(_SO))
    for name, (res, args) in {**EXPORTS, **SHARDED_EXPORTS, **MANY_LUT_EXPORTS}.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise NativeError(f"libtfhe_b200.so does not export {name}") from e
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        if not a.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous")
        return a.ctypes.data
    if isinstance(a, int):
        return a
    if hasattr(a, "data_ptr"):  # torch tensor (host pinned or device)
        return a.data_ptr()
    raise TypeError(type(a))


class Engine:
    """One tfhe_b200_ctx (one GPU).  Methods take numpy arrays (host entry points) or raw device
    pointers / torch CUDA tensors (``*_device`` entry points)."""

    def __init__(self, params: dict | Params = None, device: int = 0):
        self.lib = load_native()
        if params is None:
            params = PARAM_MESSAGE_2_CARRY_2_KS_PBS
        self.p = params if isinstance(params, Params) else Params(**params)
        h = C.c_void_p()
        self._check(self.lib.tfhe_b200_ctx_create(device, C.byref(self.p), C.byref(h)))
        self.h = h
        self.device = device
        self.many_stride = 0     # rows per ciphertext of the many-LUT entries (0: no many-LUT table uploaded)

    def _check(self, rc: int):
        if rc != 0:
            raise NativeError(self.lib.tfhe_b200_last_error().decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.tfhe_b200_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # keys -------------------------------------------------------------------------------------------
    def upload_ksk(self, ksk: np.ndarray):
        ksk = np.ascontiguousarray(ksk, dtype=np.uint64)
        self._check(self.lib.tfhe_b200_upload_ksk(self.h, _ptr(ksk), ksk.size))

    def upload_bsk_std(self, bsk: np.ndarray):
        bsk = np.ascontiguousarray(bsk, dtype=np.uint64)
        self._check(self.lib.tfhe_b200_upload_bsk_std(self.h, _ptr(bsk), bsk.size))

    def upload_seeded_ksk(self, seed16: np.ndarray, bodies: np.ndarray):
        """seeded LweKeyswitchKey: 16 seed bytes (u128 little endian) + one body word per (input key bit, level)"""
        seed16 = np.ascontiguousarray(seed16, dtype=np.uint8)
        bodies = np.ascontiguousarray(bodies, dtype=np.uint64)
        assert seed16.size == 16
        self._check(self.lib.tfhe_b200_upload_seeded_ksk(self.h, _ptr(seed16), _ptr(bodies), bodies.size))

    def upload_seeded_bsk(self, seed16: np.ndarray, bodies: np.ndarray):
        """seeded Lwe(MultiBit)BootstrapKey: 16 seed bytes + one body polynomial per GLWE row"""
        seed16 = np.ascontiguousarray(seed16, dtype=np.uint8)
        bodies = np.ascontiguousarray(bodies, dtype=np.uint64)
        assert seed16.size == 16
        self._check(self.lib.tfhe_b200_upload_seeded_bsk(self.h, _ptr(seed16), _ptr(bodies), bodies.size))

    def load_compressed_server_key(self, blob: bytes):
        """bincode-serialized shortint::CompressedServerKey (tfhe-rs 0.5): parsed on the host, masks re-drawn on the device"""
        buf = np.frombuffer(blob, dtype=np.uint8)
        self._check(self.lib.tfhe_b200_load_compressed_server_key(self.h, _ptr(buf), buf.size))

    def upload_luts(self, luts: np.ndarray):
        luts = np.ascontiguousarray(luts, dtype=np.uint64).reshape(-1, self.p.lut_len)
        self._check(self.lib.tfhe_b200_upload_luts(self.h, _ptr(luts), luts.shape[0]))
        self.n_luts = luts.shape[0]
        self.many_stride = 0

    def upload_many_luts(self, accs: np.ndarray, fn_count):
        """many-LUT accumulators (many_lut_accumulator) and their function counts; replaces the uploaded lookup tables"""
        accs = np.ascontiguousarray(accs, dtype=np.uint64).reshape(-1, self.p.lut_len)
        fn = np.ascontiguousarray(np.broadcast_to(np.asarray(fn_count, dtype=np.uint32), (accs.shape[0],)))
        self._check(self.lib.tfhe_b200_upload_many_luts(self.h, _ptr(accs), accs.shape[0], _ptr(fn)))
        self.n_luts = accs.shape[0]
        self.many_stride = int(fn.max())

    def pbs_many_batch(self, small: np.ndarray, lut_idx=None, n_iters: int | None = None) -> np.ndarray:
        """apply_many_lookup_table: (batch, S, k * N + 1), [i, f] = function f of ciphertext i (S = the largest function count)"""
        small = np.ascontiguousarray(small, dtype=np.uint64).reshape(-1, self.p.small_len)
        out = np.zeros((small.shape[0], max(self.many_stride, 1), self.p.big_len), dtype=np.uint64)
        idx = None if lut_idx is None else np.ascontiguousarray(lut_idx, dtype=np.uint32)
        if n_iters is None:
            self._check(self.lib.tfhe_b200_pbs_many_batch(self.h, _ptr(small), _ptr(idx), _ptr(out), small.shape[0]))
        else:
            self._check(self.lib.tfhe_b200_pbs_many_batch_partial(self.h, _ptr(small), _ptr(idx), _ptr(out), small.shape[0], n_iters))
        return out

    def ks_pbs_many_batch(self, cts: np.ndarray, lut_idx=None) -> np.ndarray:
        """keyswitch, then apply_many_lookup_table: (batch, S, k * N + 1)"""
        cts = np.ascontiguousarray(cts, dtype=np.uint64).reshape(-1, self.p.big_len)
        out = np.zeros((cts.shape[0], max(self.many_stride, 1), self.p.big_len), dtype=np.uint64)
        idx = None if lut_idx is None else np.ascontiguousarray(lut_idx, dtype=np.uint32)
        self._check(self.lib.tfhe_b200_ks_pbs_many_batch(self.h, _ptr(cts), _ptr(idx), _ptr(out), cts.shape[0]))
        return out

    # host-buffer hot path -------------------------------------------------------------------------------
    def keyswitch_batch(self, cts: np.ndarray) -> np.ndarray:
        cts = np.ascontiguousarray(cts, dtype=np.uint64).reshape(-1, self.p.big_len)
        out = np.empty((cts.shape[0], self.p.small_len), dtype=np.uint64)
        self._check(self.lib.tfhe_b200_keyswitch_batch(self.h, _ptr(cts), _ptr(out), cts.shape[0]))
        return out

    def pbs_batch(self, small: np.ndarray, lut_idx=None, n_iters: int | None = None) -> np.ndarray:
        small = np.ascontiguousarray(small, dtype=np.uint64).reshape(-1, self.p.small_len)
        out = np.empty((small.shape[0], self.p.big_len), dtype=np.uint64)
        idx = None if lut_idx is None else np.ascontiguousarray(lut_idx, dtype=np.uint32)
        if n_iters is None:
            self._check(self.lib.tfhe_b200_pbs_batch(self.h, _ptr(small), _ptr(idx), _ptr(out), small.shape[0]))
        else:
            self._check(self.lib.tfhe_b200_pbs_batch_partial(self.h, _ptr(small), _ptr(idx), _ptr(out), small.shape[0], n_iters))
        return out

    def ks_pbs_batch(self, cts, lut_idx=None, out=None):
        """apply_lookup_table over a batch (host buffers: numpy arrays or pinned torch tensors)."""
        if isinstance(cts, np.ndarray):
            cts = np.ascontiguousarray(cts, dtype=np.uint64).reshape(-1, self.p.big_len)
            batch = cts.shape[0]
            if out is None:
                out = np.empty_like(cts)
        else:
            batch = cts.shape[0]
        if isinstance(lut_idx, (list, tuple)):
            lut_idx = np.asarray(lut_idx, dtype=np.uint32)
        if isinstance(lut_idx, np.ndarray):
            lut_idx = np.ascontiguousarray(lut_idx, dtype=np.uint32)
        self._check(self.lib.tfhe_b200_ks_pbs_batch(self.h, _ptr(cts), _ptr(lut_idx), _ptr(out), batch))
        return out

    def pbs_ks_batch(self, small: np.ndarray, lut_idx=None) -> np.ndarray:
        """PBS -> KS order (ciphertexts under the small key), shortint/server_key/mod.rs:859-932"""
        small = np.ascontiguousarray(small, dtype=np.uint64).reshape(-1, self.p.small_len)
        out = np.empty_like(small)
        idx = None if lut_idx is None else np.ascontiguousarray(lut_idx, dtype=np.uint32)
        self._check(self.lib.tfhe_b200_pbs_ks_batch(self.h, _ptr(small), _ptr(idx), _ptr(out), small.shape[0]))
        return out

    # device-buffer hot path ---------------------------------------------------------------------------
    def ks_pbs_batch_device(self, d_in, d_idx, d_out, batch: int, stream: int | None = None):
        self._check(self.lib.tfhe_b200_ks_pbs_batch_device(self.h, _ptr(d_in), _ptr(d_idx), _ptr(d_out), batch, stream))

    def keyswitch_batch_device(self, d_in, d_small, batch: int, stream: int | None = None):
        self._check(self.lib.tfhe_b200_keyswitch_batch_device(self.h, _ptr(d_in), _ptr(d_small), batch, stream))

    def pbs_batch_device(self, d_small, d_idx, d_out, batch: int, stream: int | None = None):
        self._check(self.lib.tfhe_b200_pbs_batch_device(self.h, _ptr(d_small), _ptr(d_idx), _ptr(d_out), batch, stream))

    def pbs_many_batch_device(self, d_small, d_idx, d_out, batch: int, stream: int | None = None):
        self._check(self.lib.tfhe_b200_pbs_many_batch_device(self.h, _ptr(d_small), _ptr(d_idx), _ptr(d_out), batch, stream))

    def ks_pbs_many_batch_device(self, d_in, d_idx, d_out, batch: int, stream: int | None = None):
        self._check(self.lib.tfhe_b200_ks_pbs_many_batch_device(self.h, _ptr(d_in), _ptr(d_idx), _ptr(d_out), batch, stream))

    def set_ciphertext_modulus_log2(self, log2_q: int):
        """non-native power-of-two ciphertext modulus 2^log2_q (64 = native): PBS outputs are rounded like bootstrap.rs:318-330"""
        self._check(self.lib.tfhe_b200_set_ciphertext_modulus_log2(self.h, log2_q))

    def synchronize(self):
        self._check(self.lib.tfhe_b200_synchronize(self.h))

    def set_tuning(self, key: str, value: int):
        """kernel selection at run time (include/tfhe_b200.h: narrow_kernel, narrow_max, ks_kernel)"""
        self._check(self.lib.tfhe_b200_set_tuning(self.h, key.encode(), int(value)))

    # instrumentation -------------------------------------------------------------------------------------
    @property
    def kernel_launches(self) -> int:
        return int(self.lib.tfhe_b200_kernel_launches(self.h))

    def last_kernel_ms(self) -> tuple[float, float]:
        a, b = C.c_float(), C.c_float()
        self._check(self.lib.tfhe_b200_time_last_kernels(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def probe_fp64_tflops(self) -> float:
        v = C.c_double()
        self._check(self.lib.tfhe_b200_probe_fp64_tflops(self.device, C.byref(v)))
        return v.value
