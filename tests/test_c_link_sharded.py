"""include/tfhe_b200_sharded.h consumed from plain C (gcc -std=c99 -pedantic) and linked against libtfhe_b200.so, as tests/test_c_link.py
does for include/tfhe_b200.h: a host-language binding of the sharded program executor mirrors this header, so it must stand on its own."""
import os
import re
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def test_sharded_header_is_self_sufficient_c_and_library_links(tmp_path):
    import fhe_string_bounty_b200 as F
    so = F.build_native()
    exe = tmp_path / "link_sharded"
    cmd = ["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", str(ROOT / "include"), str(ROOT / "tests/c_link/link_sharded.c"),
           "-o", str(exe), "-L", str(so.parent), "-ltfhe_b200", f"-Wl,-rpath,{so.parent}"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "")))
    assert run.returncode == 0, run.stdout + run.stderr
    assert "2 split levels, largest share 11, 35 rows received" in run.stdout


def test_every_sharded_symbol_is_exported_and_bound():
    """every function include/tfhe_b200_sharded.h declares is exported by the library, typed by the ctypes loader and named in its C
    link test"""
    import fhe_string_bounty_b200 as F
    from fhe_string_bounty_b200 import _native
    F.build_native()
    lib = F.load_native()
    header = (ROOT / "include/tfhe_b200_sharded.h").read_text()
    declared = set(re.findall(r"\b(tfhe_b200_[a-z0-9_]+)\s*\(", header))
    declared -= {"tfhe_b200_ctx", "tfhe_b200_program", "tfhe_b200_exchange"}
    assert declared == set(_native.SHARDED_EXPORTS), sorted(declared)
    link_src = (ROOT / "tests/c_link/link_sharded.c").read_text()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} is declared but not exported"
        assert name in _native.SHARDED_EXPORTS, f"{name} is not typed in _native.SHARDED_EXPORTS"
        assert name in link_src, f"{name} is not referenced by tests/c_link/link_sharded.c"
