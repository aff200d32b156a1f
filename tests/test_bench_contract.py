"""bench.py's CPU arm (`--impl reference`): stdout is exactly ONE JSON line carrying the contract's keys; under torch.distributed.run only
rank 0 works and prints, and it uses the host's cores although the launcher exports OMP_NUM_THREADS=1 (VERDICT r1 item 2)."""
import json
import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
        "data", "config", "cpu_baseline", "e2e", "gpu_launches"}


def _one_line(out: str) -> dict:
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def _check(line: dict, n_gpus: int):
    assert KEYS <= set(line), KEYS - set(line)
    assert line["impl"] == "reference" and line["n_gpus"] == n_gpus and line["unit"] == "PBS/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == line["value"] and cb["outputs_decrypt_correctly"] is True
    assert cb["cores"] == len(os.sched_getaffinity(0))
    assert "workload" in line["config"]


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"], capture_output=True,
                       text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    _check(_one_line(r.stdout), 1)


def test_reference_arm_under_torchrun_rank0_only_all_cores():
    env = dict(os.environ, OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29533", str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    _check(_one_line(r.stdout), 2)


def test_dump_outputs_decrypt_and_repeat(tmp_path):
    """--dump-outputs writes the last timed step's output ciphertexts as float64 torus values: a second run with the same arguments
    writes the same array, and the words recovered from it decrypt to the lookup-table values of their rows"""
    import numpy as np
    import bench
    dumps = []
    for run in ("a", "b"):
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                            "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        dumps.append(np.load(tmp_path / run / "ks_pbs_out.npy"))
    a, b = dumps
    assert a.dtype == np.float64 and a.ndim == 2 and a.nbytes <= 64 << 20
    assert np.array_equal(a, b)
    assert np.all(np.abs(a) <= 0.5)
    n = _one_line(r.stdout)["config"]["batch_per_step"]
    rows = bench.dump_rows(n)
    assert a.shape[0] == len(rows)
    wl = bench.Workload("2_2")
    _, vals, idx = wl.batch(n)
    w = np.round(a * 2.0**64)
    w[w >= 2.0**63] -= 2.0**64
    words = w.astype(np.int64).view(np.uint64)
    assert words.shape[1] == wl.p.big_dim + 1
    assert wl.check(words, vals[rows], idx[rows])["ok"]
