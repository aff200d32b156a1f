"""The rotate / subtract / digit helpers of the wide blind-rotation kernels (csrc/fft_core.cuh: rot_gather, rot_sub_digit),
compiled for the CPU from the same header and checked against signed_digit_l1(+-r - o) over ties, special words, borrows, both
wrap flags, every accepted base_log and 10^7 random tuples (tests/cpu_mirror/rot_digit_check.cpp)."""
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
SRC = ROOT / "tests/cpu_mirror/rot_digit_check.cpp"


def _build_and_run(tmp_path, *defines):
    exe = tmp_path / "rot_digit_check"
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", *defines, str(SRC), "-o", str(exe)],
                   check=True, env={"PATH": "/usr/bin:/bin"})
    return subprocess.run([str(exe)], capture_output=True, text=True)


def test_rot_sub_digit_equals_signed_digit_of_the_rotated_difference(tmp_path):
    out = _build_and_run(tmp_path)
    assert out.returncode == 0, out.stdout
    assert "OK" in out.stdout


def test_checker_rejects_a_wrong_tie_rule(tmp_path):
    """The same checker against a digit whose tie goes to -B/2 instead of +B/2: the tie cases must catch it."""
    out = _build_and_run(tmp_path, "-DWRONG_TIE")
    assert out.returncode == 1, out.stdout
    assert "mismatch" in out.stdout
