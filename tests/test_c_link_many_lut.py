"""include/tfhe_b200_many_lut.h consumed from plain C (gcc -std=c99 -pedantic) and linked against libtfhe_b200.so, as tests/test_c_link.py
does for include/tfhe_b200.h."""
import os
import re
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def test_many_lut_header_is_self_sufficient_c_and_library_links(tmp_path):
    import fhe_string_bounty_b200 as F
    so = F.build_native()
    exe = tmp_path / "link_many_lut"
    cmd = ["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", str(ROOT / "include"), str(ROOT / "tests/c_link/link_many_lut.c"),
           "-o", str(exe), "-L", str(so.parent), "-ltfhe_b200", f"-Wl,-rpath,{so.parent}"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True, env=dict(os.environ))
    assert run.returncode == 0, run.stdout + run.stderr
    assert "ok: 6 symbols resolved" in run.stdout
    assert "null or empty many-LUT table" in run.stdout


def test_every_many_lut_symbol_is_exported_and_bound():
    import fhe_string_bounty_b200 as F
    from fhe_string_bounty_b200 import _native
    F.build_native()
    lib = F.load_native()
    declared = set(re.findall(r"\b(tfhe_b200_[a-z0-9_]+)\s*\(", (ROOT / "include/tfhe_b200_many_lut.h").read_text()))
    declared -= {"tfhe_b200_ctx"}
    assert declared == set(_native.MANY_LUT_EXPORTS), sorted(declared)
    link_src = (ROOT / "tests/c_link/link_many_lut.c").read_text()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} is declared but not exported"
        assert name in link_src, f"{name} is not referenced by tests/c_link/link_many_lut.c"
