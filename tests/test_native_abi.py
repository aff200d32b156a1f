"""CPU-side checks of the boundary: the library builds/loads and exports every symbol that
include/tfhe_b200.h declares; invalid parameters and the missing-GPU case fail loudly (no fallback)."""
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def native():
    import fhe_string_bounty_b200 as F
    F.build_native()
    return F


def test_header_symbols_are_exported(native):
    lib = native.load_native()
    header = (ROOT / "include" / "tfhe_b200.h").read_text()
    declared = set(re.findall(r"\b(tfhe_b200_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 15
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/tfhe_b200.h but not exported"
    from fhe_string_bounty_b200._native import EXPORTS
    assert declared == set(EXPORTS), declared ^ set(EXPORTS)


def test_no_cpu_fallback(native):
    """without a visible device Engine() raises NativeError; the child process hides every GPU, so this holds on GPU machines too"""
    import os
    import subprocess
    import sys
    code = "import fhe_string_bounty_b200 as F\ntry:\n    F.Engine()\nexcept F.NativeError:\n    print('NativeError')\n"
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=300,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0 and r.stdout.strip() == "NativeError", r.stdout + r.stderr


def test_rejects_unsupported_params(native):
    import ctypes as C
    lib = native.load_native()
    bad = dict(native.PARAM_MESSAGE_2_CARRY_2_KS_PBS, poly_size=1024)
    p = native.Params(**bad)
    h = C.c_void_p(123)
    assert lib.tfhe_b200_ctx_create(0, C.byref(p), C.byref(h)) != 0
    assert h.value is None  # out pointer nulled first (c_api/shortint/server_key/pbs.rs:26-28 convention)
    assert b"poly_size" in lib.tfhe_b200_last_error()
    assert lib.tfhe_b200_ctx_create(0, None, C.byref(h)) != 0
    assert lib.tfhe_b200_ctx_create(0, C.byref(p), None) != 0


def test_level_planner_covers_every_width(native):
    """the dispatcher's cut of a level into (4 per SM, 3 per SM, narrow tail) launches: every ciphertext exactly once, each part within
    what its kernel takes, never more waves than the all-4-per-SM cut, and the cuts the measured wave times favour"""
    import ctypes as C
    lib = native.load_native()
    sms = 148

    def plan(batch, narrow=2 * sms, cluster=1):
        out = (C.c_size_t * 3)()
        lib.tfhe_b200_plan_classic_level(batch, sms, narrow, cluster, out)
        return tuple(out)

    cost = {4: 7.2, 3: 5.49}
    for batch in list(range(1, 1400)) + [1920, 1984, 4096, 8192, 16384, 65536, 65537]:
        n4, n3, tail = plan(batch)
        assert n4 + n3 + tail == batch
        assert tail <= 2 * sms
        assert n4 % (4 * sms) == 0 or n3 + tail == 0          # only the last part may end inside a wave
        assert n3 % (3 * sms) == 0 or tail == 0
        waves = lambda n, per: -(-n // (per * sms))
        t = waves(n4, 4) * cost[4] + waves(n3, 3) * cost[3] + (0 if tail == 0 else 1.84 if tail <= sms // 2 else 2.75 if tail <= sms else 4.37)
        assert t <= waves(batch, 4) * cost[4] + 1e-9, (batch, n4, n3, tail)
    assert plan(74) == (0, 0, 74) and plan(296) == (0, 0, 296)
    assert plan(297) == (0, 297, 0) and plan(444) == (0, 444, 0)
    assert plan(445) == (445, 0, 0) and plan(592) == (592, 0, 0)
    assert plan(592 + 30) == (592, 0, 30)
    assert plan(592 + 200) == (0, 792, 0)                        # two waves of three beat a wave of four plus a two-per-SM tail
    assert plan(1024) == (592, 432, 0)
    assert plan(8192) == (8192, 0, 0)
    # no narrow kernels: everything to the wide kernel, whose launcher picks the instance
    assert plan(100, narrow=0) == (100, 0, 0) and plan(1000, narrow=0) == (1000, 0, 0)
    # a narrow kernel limited to one ciphertext per SM
    assert plan(200, narrow=sms) == (0, 200, 0) and plan(592 + 100, narrow=sms) == (592, 0, 100)


def test_cpu_mirror_of_warp_fft(tmp_path):
    """tests/cpu_mirror/fft_mirror.cpp emulates the 32 lanes of the warp FFT from the SAME header the
    kernels compile (fft_core.cuh) and checks it against the DFT definition."""
    import subprocess
    exe = tmp_path / "fft_mirror"
    subprocess.run(["g++", "-O1", "-std=c++17", "-ffp-contract=off", str(ROOT / "tests/cpu_mirror/fft_mirror.cpp"), "-o", str(exe)],
                   check=True, env={"PATH": "/usr/bin:/bin"})
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert "OK" in out.stdout


def test_cpu_mirror_of_two_warp_fft(tmp_path):
    """tests/cpu_mirror/fft16_mirror.cpp emulates the 64 threads of the 16 x 4 x 16 FFT of the v4 blind-rotation kernel from the
    SAME header the kernel compiles (fft16_core.cuh): DFT definition, frequency map, round trip, bank-conflict-free and
    region-confined exchange addressing."""
    import subprocess
    exe = tmp_path / "fft16_mirror"
    subprocess.run(["g++", "-O1", "-std=c++17", "-ffp-contract=off", str(ROOT / "tests/cpu_mirror/fft16_mirror.cpp"), "-o", str(exe)],
                   check=True, env={"PATH": "/usr/bin:/bin"})
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert "OK" in out.stdout


def test_cpu_mirror_of_four_warp_fft(tmp_path):
    """tests/cpu_mirror/fft8_mirror.cpp: the 128-thread x 8-point FFT of the experimental narrow-level kernel (fft8_core.cuh)."""
    import subprocess
    exe = tmp_path / "fft8_mirror"
    subprocess.run(["g++", "-O1", "-std=c++17", "-ffp-contract=off", str(ROOT / "tests/cpu_mirror/fft8_mirror.cpp"), "-o", str(exe)],
                   check=True, env={"PATH": "/usr/bin:/bin"})
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert "OK" in out.stdout


def test_parameter_tables_match_the_oracle_and_the_engine_envelope():
    """The product's parameter tables (classic_params / multi_bit_params) against the oracle's independently typed copies of
    shortint/parameters/{mod,multi_bit}.rs, and every set inside the envelope tfhe_b200_ctx_create accepts (c_api.cu check_params)."""
    import fhe_string_bounty_b200 as F
    from fhe_string_bounty_b200._native import _CLASSIC_SETS, _MULTI_BIT_SETS
    from oracle import oracle as O
    assert len(_CLASSIC_SETS) == 36 and len(_MULTI_BIT_SETS) == 6
    assert F.classic_params("2_2") == dict(F.PARAM_MESSAGE_2_CARRY_2_KS_PBS)
    assert F.multi_bit_params("2_2_g3") == dict(F.PARAM_MULTI_BIT_MESSAGE_2_CARRY_2_GROUP_3_KS_PBS)
    fields = ("lwe_dim", "glwe_dim", "poly_size", "pbs_base_log", "pbs_level", "ks_base_log", "ks_level", "grouping_factor", "msg_mod", "carry_mod")
    for name in O.OTHER_CLASSIC_SETS:
        op, mine = O.params(name), F.classic_params(name)
        assert all(getattr(op, f) == mine[f] for f in fields), name
    for name in O.OTHER_MULTI_BIT_SETS:
        op, mine = O.params(name), F.multi_bit_params(name.replace("multibit_", ""))
        assert all(getattr(op, f) == mine[f] for f in fields), name
    shapes = {(256, 5), (512, 3), (512, 2), (1024, 2), (2048, 1), (4096, 1), (8192, 1), (16384, 1), (32768, 1)}
    for name, t in list(_CLASSIC_SETS.items()) + list(_MULTI_BIT_SETS.items()):
        n, k, N, pb, pl, kb, kl = t[:7]
        assert (N, k) in shapes and 2 <= kb <= 7 and kb * kl <= 31 and 2 <= pb <= 30 and pb * pl <= 52 and n <= 4096, name


def test_cpu_mirror_of_the_16x16_and_16x16x16_ffts(tmp_path):
    """tests/cpu_mirror/fft16x_mirror.cpp: the 256-point FFT of pbs_n512.cu (16 threads) and the 4096-point FFT of pbs_n8192.cu (256
    threads), emulated thread by thread from the slot functions and twiddle tables the kernels use (csrc/fft16x_slots.cuh): forward ==
    definition at the documented frequency map, inverse(forward) == M x, exchanges injective and bank-conflict free."""
    import subprocess
    exe = tmp_path / "fft16x_mirror"
    subprocess.run(["g++", "-O1", "-std=c++17", "-ffp-contract=off", str(ROOT / "tests/cpu_mirror/fft16x_mirror.cpp"), "-o", str(exe)],
                   check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.strip().endswith("OK"), out.stdout + out.stderr
