#!/usr/bin/env python
"""bench.py -- batched KS-PBS throughput on B200 (BASELINE.json configs[1]) and the CPU reference arm.

    python bench.py --gpus N --steps K --warmup W            # this engine (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs (see dump_outputs)

A "step" is one pass of the hot path -- keyswitch + programmable bootstrap with per-ciphertext lookup table -- over one batch of
`--batch` independent LWE ciphertexts per GPU at PARAM_MESSAGE_2_CARRY_2_KS_PBS.  `value` is device-timed whole-job KS-PBS/s with
inputs resident in HBM; `e2e` is the same metric through the host-buffer C-ABI call (tfhe_b200_ks_pbs_batch) with pinned host inputs
and outputs, copies inside the timed region.

Keys are REAL seeded keys and the batch holds real encryptions (generated with the CPU oracle, which here is only the key generator /
encryptor / decryptor, i.e. the checker): after the timed region every output ciphertext of the timed configuration -- same context,
same batch size, same kernel selection -- is decrypted and compared with its lookup-table value (`validation`).  The string
operations are validated the same way against clear-text semantics.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SETS = {
    "2_2": dict(oracle="2_2", name="PARAM_MESSAGE_2_CARRY_2_KS_PBS", config="configs[1]", kernel="pbs_classic_kernel_v4"),
    "multibit": dict(oracle="multibit_2_2_g3", name="PARAM_MULTI_BIT_MESSAGE_2_CARRY_2_GROUP_3_KS_PBS", config="configs[4]",
                     kernel="pbs_multibit_kernel_v4"),
}
LUT_FUNCS = [lambda x, a=a, b=b: (a * x + b) % 16 for a, b in
             [(1, 0), (3, 1), (5, 2), (7, 3), (9, 4), (11, 5), (13, 6), (15, 7), (1, 8), (3, 9), (5, 10), (7, 11), (9, 12), (11, 13), (13, 14), (15, 15)]]


def flop_per_pbs(p) -> float:
    """SURVEY.md 8(d): steps * ((k+1)(l+1)(5 M log2 M + 6 M) + (k+1)^2 l M 8) [+ the multi-bit combine: (2^g - 1) (k+1)^2 l M 14 per group]"""
    M, k1, l = p.poly_size // 2, p.glwe_dim + 1, p.pbs_level
    per = k1 * (l + 1) * (5 * M * math.log2(M) + 6 * M) + k1 * k1 * l * M * 8
    if p.grouping_factor:
        return (p.lwe_dim // p.grouping_factor) * (per + ((1 << p.grouping_factor) - 1) * k1 * k1 * l * M * 14)
    return p.lwe_dim * per


def bsk_fourier_bytes(p) -> int:
    n_ggsw = p.lwe_dim if not p.grouping_factor else (p.lwe_dim // p.grouping_factor) << p.grouping_factor
    return n_ggsw * p.pbs_level * (p.glwe_dim + 1) ** 2 * (p.poly_size // 2) * 16


def host_cores() -> int:
    """the cores this process may run on -- NOT omp_get_max_threads(): torch.distributed.run exports OMP_NUM_THREADS=1"""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def _clock_sampler(stop, samples, device_index):
    q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    while not stop.is_set():
        try:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(device_index)],
                                 capture_output=True, text=True, timeout=5).stdout.strip()
            if out:
                samples.append([s.strip() for s in out.split(",")])
        except Exception:
            pass
        stop.wait(0.2)


def _summarise_clocks(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
    sm = sorted(float(s[0]) for s in samples if s[0].replace(".", "").isdigit())
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    reasons = [n for i, n in enumerate(names) if any(len(s) > 3 + i and s[3 + i].lower().startswith("active") for s in samples)]
    return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(samples[0][1]) if samples[0][1].replace(".", "").isdigit() else None,
            "power_w_max": max((float(s[2]) for s in samples if s[2].replace(".", "").isdigit()), default=None),
            "samples": len(samples), "reasons": reasons}


def _peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        return json.loads(f.read_text()), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


class Workload:
    """Seeded client / server keys of one parameter set, 16 lookup tables and a tile of real encryptions (all from the CPU oracle: key
    generation, encryption and decryption are client-side operations the engine does not have)."""

    def __init__(self, which: str, n_base: int = 256):
        from oracle import oracle as O
        self.O = O
        self.p = O.params(SETS[which]["oracle"])
        self.ck = O.ClientKey(self.p, 0xB200 + 1)
        self.sk = O.ServerKey(self.ck, 0xB300 + 1)
        self.luts = np.stack([self.sk.generate_lookup_table(f)[0] for f in LUT_FUNCS])
        rng = np.random.default_rng(0xB200)
        self.base_vals = rng.integers(0, 16, size=n_base)
        self.base_cts = self.ck.encrypt_batch(self.base_vals)

    def batch(self, n: int, offset: int = 0):
        """n ciphertexts (the tile repeated), their clear values and per-ciphertext LUT indices"""
        nb = len(self.base_vals)
        sel = (np.arange(n) + offset) % nb
        idx = ((np.arange(n) * 5 + np.arange(n) // nb + offset) % 16).astype(np.uint32)
        return self.base_cts[sel], self.base_vals[sel], idx

    def expected(self, vals, idx):
        return np.array([LUT_FUNCS[i](int(v)) for v, i in zip(vals, idx)])

    def check(self, out_cts, vals, idx) -> dict:
        got = self.ck.decrypt_batch(np.ascontiguousarray(out_cts))
        want = self.expected(vals, idx)
        bad = int((got != want).sum())
        return {"checked": int(len(want)), "mismatches": bad, "ok": bad == 0}


class CpuReference:
    """The CPU oracle (restatement of the reference's KS-PBS, one ciphertext per OpenMP thread, the structure of
    tfhe/benches/core_crypto/pbs_bench.rs:512-536) on the same seeded keys and ciphertexts, with an EXPLICIT thread count."""

    def __init__(self, wl: Workload, max_cts: int, threads: int = 0):
        import ctypes as C
        self.C, self.L, self.wl = C, wl.O.lib(), wl
        self.cts, self.vals, self.idx = wl.batch(max_cts)
        self.cts = np.ascontiguousarray(self.cts)
        self.out = np.zeros_like(self.cts)
        self.cores = threads or host_cores()

    def run(self, n_cts: int):
        C, sk = self.C, self.wl.sk
        t0 = time.perf_counter()
        used = self.L.orc_ks_pbs_batch(C.byref(sk.p), sk.ksk, sk.fourier, self.wl.luts, self.idx.ctypes.data_as(C.c_void_p),
                                       self.cts[:n_cts], self.out[:n_cts], None, n_cts, self.cores)
        return time.perf_counter() - t0, used

    def validate(self, n_cts: int) -> bool:
        return self.wl.check(self.out[:n_cts], self.vals[:n_cts], self.idx[:n_cts])["ok"]


DUMP_ROWS = 2048        # 2048 x 2049 words x 8 B = 34 MB of float64 for the 2_2 and multi-bit sets


def dump_rows(n: int) -> np.ndarray:
    """the rows dump_outputs keeps of an n-ciphertext batch: all of them, or a fixed, seeded sample of DUMP_ROWS in batch order"""
    return np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0xD0).choice(n, DUMP_ROWS, replace=False))


def dump_outputs(out_dir: str, cts: np.ndarray):
    """Writes out_dir/ks_pbs_out.npy: the output LWE ciphertexts of the last timed step, rows dump_rows(batch), as float64 torus values
    (signed word / 2^64, in [-0.5, 0.5]).  The inputs are seeded, so two builds run with the same arguments can be compared row for row;
    the low bits of each word carry the FFT's rounding, so the comparison wants a tolerance rather than equality."""
    torus = np.ascontiguousarray(cts[dump_rows(cts.shape[0])]).view(np.int64).astype(np.float64) / 2.0**64
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / "ks_pbs_out.npy", torus)


def cpu_reference_rate(wl: Workload, n_cts: int):
    ref = CpuReference(wl, n_cts)
    ref.run(min(n_cts, ref.cores))          # warm-up: page in the Fourier key, spin up the OpenMP team
    dt, used = ref.run(n_cts)
    ok = ref.validate(min(n_cts, 256))
    return n_cts / dt, used, dt, ok


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = Workload(args.params)
    cores = host_cores()
    per_step = cores * 32               # about 0.8 s of work per step
    ref = CpuReference(wl, per_step, cores)
    total_t, used = 0.0, cores
    for s in range(args.warmup + args.steps):
        dt, used = ref.run(per_step)
        if s >= args.warmup:
            total_t += dt
    ok = ref.validate(min(per_step, 256))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ref.out[:per_step])
    value = per_step * args.steps / total_t
    line = {
        "impl": "reference", "metric": "batched KS-PBS throughput", "value": value, "unit": "PBS/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_t / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{SETS[args.params]['name']} batched KS-PBS ({SETS[args.params]['config']})", "batch_per_step": per_step,
                   "note": "throughput metric: each step is a bounded sample (cores x 32 ciphertexts) of the GPU arm's workload; the "
                           "reference Rust crate cannot be built here (no cargo), this is the CPU oracle port of its algorithm on all "
                           "host cores (thread count passed explicitly, OMP_NUM_THREADS is not inherited)"},
        "cpu_baseline": {"value": value, "unit": "PBS/s", "cores": used, "kind": "port",
                         "sample": f"{per_step} KS-PBS per step x {args.steps} steps, one ciphertext per OpenMP thread, real seeded keys",
                         "outputs_decrypt_correctly": ok},
        "e2e": {"value": value, "unit": "PBS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


_JSON_FD = None


def emit(line: dict):
    """the JSON line, on the process's original stdout (see main)"""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def run_param_sweep(args):
    """--param-sweep: KS-PBS/s of other classic parameter sets (SURVEY 8(f) N4) on one GPU next to the CPU oracle on the same box.
    Device-resident inputs, CUDA events on the launching stream, random key words (timing only: parity of these sets is
    tests/test_gpu_param_sets.py).  One JSON line; not the headline metric."""
    rows = param_sweep_rows(args.param_sweep.split(","), args.cpu_sample != 0, 0)
    emit({"metric": "KS-PBS throughput per classic parameter set (1 GPU, device-resident)", "unit": "PBS/s", "sets": rows})


def param_sweep_rows(names, with_cpu: bool, device: int):
    import ctypes as C
    import torch
    import fhe_string_bounty_b200 as F
    torch.cuda.set_device(device)
    sms = torch.cuda.get_device_properties(device).multi_processor_count
    rows = []
    for name in names:
        p = F.Params(**F.classic_params(name))
        eng = F.Engine(p, device=device)
        rng = np.random.default_rng(0xB200)
        ksk = rng.integers(0, 2**64, size=p.ksk_len, dtype=np.uint64)
        bsk = rng.integers(0, 2**64, size=p.bsk_len, dtype=np.uint64)
        luts = rng.integers(0, 2**64, size=(4, p.lut_len), dtype=np.uint64)
        eng.upload_ksk(ksk)
        eng.upload_bsk_std(bsk)
        eng.upload_luts(luts)
        small_n = p.poly_size <= 8192
        B = (8 if small_n else 2) * sms
        d_in = torch.randint(-2**63, 2**63 - 1, (B, p.big_len), dtype=torch.int64, device="cuda")
        d_idx = (torch.arange(B, device="cuda", dtype=torch.int32) % 4).contiguous()
        d_out = torch.empty_like(d_in)
        ts = torch.cuda.Stream()
        torch.cuda.set_stream(ts)
        eng.ks_pbs_batch_device(d_in, d_idx, d_out, B, ts.cuda_stream)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3 if small_n else 1
        ev0.record()
        for _ in range(reps):
            eng.ks_pbs_batch_device(d_in, d_idx, d_out, B, ts.cuda_stream)
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / reps
        ks_ms, pbs_ms = eng.last_kernel_ms()
        eng.close()
        del d_in, d_out
        torch.cuda.empty_cache()
        flop = flop_per_pbs(p)
        row = {"params": f"PARAM_MESSAGE_{name.replace('_', '_CARRY_')}_KS_PBS", "N": p.poly_size, "k": p.glwe_dim, "pbs_level": p.pbs_level,
               "batch": B, "ms": ms, "keyswitch_ms": ks_ms, "pbs_ms": pbs_ms, "ks_pbs_per_s": B / (ms * 1e-3), "flop_per_pbs": flop,
               "pbs_tflops": B * flop / (pbs_ms * 1e-3) / 1e12}
        if with_cpu:
            from oracle import oracle as O
            L, op = O.lib(), O.params(name)
            cores = host_cores()
            n_cpu = cores * (2 if small_n else 1)
            f = L.orc_fourier_bsk_new(C.byref(op), bsk)
            cts = rng.integers(0, 2**64, size=(n_cpu, op.big_dim + 1), dtype=np.uint64)
            out = np.zeros_like(cts)
            idx = (np.arange(n_cpu) % 4).astype(np.uint32)
            call = lambda n: L.orc_ks_pbs_batch(C.byref(op), ksk, f, luts, idx.ctypes.data_as(C.c_void_p), cts[:n], out[:n], None, n, cores)
            call(min(n_cpu, cores))
            t0 = time.perf_counter()
            used = call(n_cpu)
            dt = time.perf_counter() - t0
            L.orc_fourier_bsk_free(f)
            row["cpu_port_ks_pbs_per_s"] = n_cpu / dt
            row["cpu_cores"] = used
            row["gpu_over_cpu"] = row["ks_pbs_per_s"] / row["cpu_port_ks_pbs_per_s"]
        rows.append(row)
    return rows


def _timed_ops(fn, reps, world):
    """ops/s of fn() through host buffers (wall clock around reps calls, each ending in its own device -> host copy); max over ranks"""
    import torch
    import torch.distributed as dist
    fn()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t[0])
    return reps / dt


def bench_string_ops(eng, wl: Workload, rank, world, exchange):
    """FheString ops per second (BASELINE.json configs[0], [2], [3]) through the host layer: encrypted strings leave from page-locked host
    memory, every tree level's launches, the narrow-end exchange between the ranks (the engine's peer-memory kernel, or NCCL with
    --exchange nccl) and the finishing levels stay on the device, the result block comes back to the host -- all inside the timed
    region.  Every operation's decrypted result is checked against clear text once, outside the timing."""
    import torch
    import fhe_string_bounty_b200 as F
    from fhe_string_bounty_b200 import multi_gpu as MG
    from fhe_string_bounty_b200.host import Program
    from oracle import radix as R
    params = dict(F.PARAM_MESSAGE_2_CARRY_2_KS_PBS)
    p, ck = eng.p, wl.ck
    rng = np.random.default_rng(77)              # same on every rank (the operands are replicated, the work is sharded)
    comm = MG.DeviceComm(eng, rank=rank, world=world, exchange=exchange)
    out, checks = {}, {}
    _pinned = []

    def pin(arr):
        """page-locked copy of a host array (the e2e contract: inputs leave from pinned host memory)"""
        t = torch.from_numpy(np.ascontiguousarray(arr).view(np.int64)).pin_memory()
        _pinned.append(t)
        return t.numpy().view(np.uint64)

    def run_pinned(prog, ins):
        """single-GPU program through host buffers, both of them page-locked"""
        key = id(prog)
        if key not in run_pinned.out:
            run_pinned.out[key] = pin(np.zeros((prog.n_outputs, p.big_len), dtype=np.uint64))
        return prog.run(eng, ins, out=run_pinned.out[key])
    run_pinned.out = {}

    rand_str = lambda n: bytes(rng.integers(ord("a"), ord("z") + 1, size=n).tolist())
    dec = ck.decrypt_message_and_carry
    # config 1: eq of two 8-char strings (equal: the full tree is exercised either way)
    s8 = rand_str(8)
    a8, b8 = pin(R.encrypt_string(ck, s8)), pin(R.encrypt_string(ck, s8))
    c8 = pin(R.encrypt_string(ck, s8[:5] + b"#" + s8[6:]))
    checks["eq_8char"] = dec(MG.sharded_eq(comm, params, a8, b8, 8)) == 1 and dec(MG.sharded_eq(comm, params, a8, c8, 8)) == 0
    out["eq_8char_ops_per_s"] = _timed_ops(lambda: MG.sharded_eq(comm, params, a8, b8, 8), 20, world)
    # config 3: contains / find, 256-char haystack, 16-char pattern taken from offset 201
    hs = rand_str(256)
    ps = hs[201:217]
    hay, pat = pin(R.encrypt_string(ck, hs)), pin(R.encrypt_string(ck, ps))
    nopat = pin(R.encrypt_string(ck, b"0123456789ABCDEF"))
    checks["contains_256_16"] = dec(MG.sharded_contains(comm, params, hay, pat, 256, 16)) == 1 and \
        dec(MG.sharded_contains(comm, params, hay, nopat, 256, 16)) == 0
    out["contains_256_16_ops_per_s"] = _timed_ops(lambda: MG.sharded_contains(comm, params, hay, pat, 256, 16), 3, world)
    r = MG.sharded_find(comm, params, hay, pat, 256, 16)
    checks["find_256_16"] = (dec(r[0]), R.decrypt_radix(ck, r[1:])) == (1, hs.find(ps))
    if not checks["find_256_16"]:
        out["find_256_16_got_want"] = [[int(dec(r[0])), int(R.decrypt_radix(ck, r[1:]))], [1, hs.find(ps)]]
    out["find_256_16_ops_per_s"] = _timed_ops(lambda: MG.sharded_find(comm, params, hay, pat, 256, 16), 3, world)
    # config 4: case conversion of a 1024-char string (each rank keeps its own converted chars: no exchange on the path)
    s1k = bytes(rng.integers(0x20, 0x7F, size=1024).tolist())
    e1k = pin(R.encrypt_string(ck, s1k))
    low = MG.sharded_case(comm, params, "to_lowercase", e1k, 1024, gather=False)
    c0, c1 = MG.shard_range(1024, rank, min(world, 1024))
    checks["to_lowercase_1024"] = R.decrypt_string(ck, low) == s1k.lower()[c0:c1]
    out["to_lowercase_1024_ops_per_s"] = _timed_ops(lambda: MG.sharded_case(comm, params, "to_lowercase", e1k, 1024, gather=False), 3, world)
    # throughput mode: independent string pairs share each tree level's launches (each rank takes its own share of pairs)
    n_pairs = 512
    many = Program("string_eq_many", (8, 8, n_pairs), params=params)
    pairs = pin(rng.integers(0, 2**64, size=(many.n_inputs, p.big_len), dtype=np.uint64))
    pairs[:64] = np.concatenate([a8, b8])         # pair 0 real and equal, pair 1..: random words (timing only)
    checks["eq_8char_batched"] = dec(run_pinned(many, pairs)[0]) == 1
    out["eq_8char_batched_ops_per_s"] = world * n_pairs * _timed_ops(lambda: run_pinned(many, pairs), 3, world)
    out["eq_8char_batch"] = {"pairs_per_rank": n_pairs, "pbs": many.n_pbs, "levels": many.level_widths}
    manyp = Program("string_eq_many_packed", (8, 8, n_pairs), params=params)    # one PBS per pair of blocks (comparator.rs:193-221)
    out["eq_8char_batched_packed_ops_per_s"] = world * n_pairs * _timed_ops(lambda: run_pinned(manyp, pairs), 3, world)
    out["eq_8char_batch_packed"] = {"pairs_per_rank": n_pairs, "pbs": manyp.n_pbs, "levels": manyp.level_widths}
    if world == 1:
        ins_c = pin(np.concatenate([hay, pat]))
        cp = Program("string_contains_packed", (256, 16), params=params)
        checks["contains_256_16_packed"] = dec(run_pinned(cp, ins_c)[0]) == 1
        out["contains_256_16_packed_ops_per_s"] = _timed_ops(lambda: run_pinned(cp, ins_c), 3, world)
        out["contains_256_16_packed_pbs"] = cp.n_pbs
        findp = Program("string_find_packed", (256, 16), params=params)
        r = run_pinned(findp, ins_c)
        checks["find_256_16_packed"] = (dec(r[0]), R.decrypt_radix(ck, r[1:])) == (1, hs.find(ps))
        out["find_256_16_packed_ops_per_s"] = _timed_ops(lambda: run_pinned(findp, ins_c), 3, world)
        out["find_256_16_packed_pbs"] = findp.n_pbs
        up = Program("string_to_uppercase", (1024,), params=params)
        checks["to_uppercase_1024"] = R.decrypt_string(ck, run_pinned(up, e1k)) == s1k.upper()
        out["to_uppercase_1024_ops_per_s"] = _timed_ops(lambda: run_pinned(up, e1k), 3, world)
        eic = Program("string_eq_ignore_case", (1024, 1024), params=params)
        two = pin(np.concatenate([e1k, R.encrypt_string(ck, s1k.swapcase())]))
        checks["eq_ignore_case_1024"] = dec(run_pinned(eic, two)[0]) == 1
        out["eq_ignore_case_1024_ops_per_s"] = _timed_ops(lambda: run_pinned(eic, two), 2, world)
        out["eq_ignore_case_1024_pbs"] = eic.n_pbs
    out["pbs_counts"] = {"eq_8char": Program("string_eq", (8, 8), params=params).n_pbs,
                         "contains_256_16": Program("string_contains", (256, 16), params=params).n_pbs,
                         "find_256_16": Program("string_find", (256, 16), params=params).n_pbs,
                         "to_lowercase_1024": Program("string_to_lowercase", (1024,), params=params).n_pbs}
    out["decrypted_results_correct"] = {k: bool(v) for k, v in checks.items()}
    out["exchange"] = "none (1 rank)" if world == 1 else ("engine peer-memory kernel over CUDA IPC / NVLink (csrc/exchange.cu)" if comm.peer is not None else "NCCL")
    out["note"] = ("page-locked host buffers in, result block out; eq shards chars, contains / find shard windows, to_lowercase shards chars "
                   "(each rank keeps its converted chars); one exchange of 1 (eq, contains) / 1 + 4 (find) LWE blocks per rank at the narrow end")
    comm.close()
    return out


def bench_multibit_compare(local, rank, world, exchange):
    """BASELINE.json configs[4]: lexicographic lt / le on 128-char strings with PARAM_MULTI_BIT_MESSAGE_2_CARRY_2_GROUP_3_KS_PBS.  Two
    numbers: the comparison SHARDED over the ranks (chars split, one gather of the ranks' sign blocks, sign tree on every rank: latency
    of one comparison) and whole comparisons as independent replicas (ops/s = ranks x one rank's rate)."""
    import torch
    import fhe_string_bounty_b200 as F
    from fhe_string_bounty_b200 import multi_gpu as MG
    from fhe_string_bounty_b200.host import Program
    from oracle import radix as R
    wl = Workload("multibit", n_base=16)
    params = dict(F.PARAM_MULTI_BIT_MESSAGE_2_CARRY_2_GROUP_3_KS_PBS)
    eng = F.Engine(params, device=local)
    eng.upload_ksk(wl.sk.ksk)
    eng.upload_bsk_std(wl.sk.bsk)
    ck, dec = wl.ck, wl.ck.decrypt_message_and_carry
    rng = np.random.default_rng(78)
    a = bytes(rng.integers(0x20, 0x7F, size=128).tolist())
    b = a[:97] + bytes([a[97] + 1 if a[97] < 0x7E else 0x20]) + a[98:]
    pin = lambda arr: torch.from_numpy(np.ascontiguousarray(arr).view(np.int64)).pin_memory().numpy().view(np.uint64)
    ea, eb = pin(R.encrypt_string(ck, a)), pin(R.encrypt_string(ck, b))
    comm = MG.DeviceComm(eng, rank=rank, world=world, exchange=exchange)
    out, checks = {}, {}
    for op, want in (("lt", a < b), ("le", a <= b)):
        checks[op + "_sharded"] = dec(MG.sharded_compare(comm, params, op, ea, eb, 128)) == int(want) and \
            dec(MG.sharded_compare(comm, params, op, ea, ea, 128)) == int(op == "le")
        rate = _timed_ops(lambda: MG.sharded_compare(comm, params, op, ea, eb, 128), 5, world)
        out[op + "_128char_multibit_sharded_ms"] = 1e3 / rate
        out[op + "_128char_multibit_sharded_ops_per_s"] = rate
        prog = Program("string_" + op, (128, 128), params=params)
        ins = pin(np.concatenate([ea, eb]))
        checks[op + "_replica"] = dec(prog.run(eng, ins)[0]) == int(want)
        rate = _timed_ops(lambda: prog.run(eng, ins), 5, world)
        out[op + "_128char_multibit_replica_ms"] = 1e3 / rate
        out[op + "_128char_multibit_replicas_ops_per_s"] = world * rate
        out[op + "_128char_pbs"] = prog.n_pbs
    out["decrypted_results_correct"] = {k: bool(v) for k, v in checks.items()}
    out["note"] = ("config 5: 'sharded' = one comparison over all ranks (latency), 'replicas' = every rank compares its own pair (throughput); "
                   "512 PBS in 10 levels [256, 128, ..., 1, 1] unsharded")
    comm.close()
    eng.close()
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    import fhe_string_bounty_b200 as F

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL writes its version banner (any NCCL_DEBUG level from VERSION up, which the GPU boxes set) and its warnings to stdout by
        # default: send them to stderr so that stdout stays the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    B = args.batch
    meta = SETS[args.params]
    p = F.Params(**(F.PARAM_MULTI_BIT_MESSAGE_2_CARRY_2_GROUP_3_KS_PBS if args.params == "multibit" else F.PARAM_MESSAGE_2_CARRY_2_KS_PBS))
    FLOP, BSK_BYTES = flop_per_pbs(p), bsk_fourier_bytes(p)
    KSK_BYTES = p.glwe_dim * p.poly_size * p.ks_level * p.small_len * 8
    CT_BYTES, SMALL_BYTES = p.big_len * 8, p.small_len * 8
    wl = Workload(args.params)                   # same seeds on every rank: keys are replicated, work is sharded
    eng = F.Engine(p, device=local)
    eng.upload_ksk(wl.sk.ksk)
    eng.upload_bsk_std(wl.sk.bsk)
    eng.upload_luts(wl.luts)
    sms = torch.cuda.get_device_properties(local).multi_processor_count

    cts, vals, idx = wl.batch(B, offset=17 * rank)
    d_in = torch.from_numpy(cts.view(np.int64)).cuda()
    d_idx = torch.from_numpy(idx.view(np.int32)).cuda()
    d_out = torch.empty_like(d_in)
    # a non-default torch stream: handle 0 would mean "the context's own stream" to the C ABI, and
    # torch.cuda.Event only sees the stream it is recorded on
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    def step():
        eng.ks_pbs_batch_device(d_in, d_idx, d_out, B, stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    stop, samples = threading.Event(), []
    sampler = threading.Thread(target=_clock_sampler, args=(stop, samples, local), daemon=True)
    sampler.start()
    launches0 = eng.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ks_ms_sum = pbs_ms_sum = 0.0
    barrier()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = eng.kernel_launches - launches0
    # the timed configuration's outputs, decrypted: every ciphertext of the batch against its lookup-table value
    h_last = d_out.cpu().numpy().view(np.uint64)
    validation = wl.check(h_last, vals, idx)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, h_last)
    # per-kernel durations of the dominant kernel, measured live (CUDA events on the launching stream)
    for _ in range(min(args.steps, 5)):
        step()
        torch.cuda.synchronize()
        k, q = eng.last_kernel_ms()
        ks_ms_sum += k
        pbs_ms_sum += q
    n_k = min(args.steps, 5)
    ks_ms, pbs_ms = ks_ms_sum / n_k, pbs_ms_sum / n_k
    stop.set()
    sampler.join(timeout=2)

    # e2e through the host-buffer C-ABI entry point, pinned host memory, copies inside the timed region
    h_in = torch.from_numpy(cts.view(np.int64)).pin_memory()
    h_idx = torch.from_numpy(idx.view(np.int32)).pin_memory()
    h_out = torch.empty((B, p.big_len), dtype=torch.int64).pin_memory()
    e2e_steps = max(2, min(args.steps, 5))
    eng.ks_pbs_batch(h_in, h_idx, h_out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        eng.ks_pbs_batch(h_in, h_idx, h_out)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_validation = wl.check(h_out.numpy().view(np.uint64), vals, idx)

    # config 2 names 4096 ... 65536 evaluations: the same step at the other batch sizes (device-timed, 2 steps each)
    batch_sweep = []
    if args.batch_sweep:
        wave = (3 if p.grouping_factor else 4) * sms
        for b2 in [int(x) for x in args.batch_sweep.split(",")]:
            c2, v2, i2 = wl.batch(b2, offset=3 + rank)
            di, dx = torch.from_numpy(c2.view(np.int64)).cuda(), torch.from_numpy(i2.view(np.int32)).cuda()
            do = torch.empty_like(di)
            eng.ks_pbs_batch_device(di, dx, do, b2, stream)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(2):
                eng.ks_pbs_batch_device(di, dx, do, b2, stream)
            e1.record()
            torch.cuda.synchronize()
            t_ms = e0.elapsed_time(e1) / 2
            ok = wl.check(do[:: max(1, b2 // 512)].cpu().numpy().view(np.uint64), v2[:: max(1, b2 // 512)], i2[:: max(1, b2 // 512)])["ok"]
            batch_sweep.append({"batch_per_gpu": b2, "ms_per_step": t_ms, "pbs_per_s_per_gpu": b2 / (t_ms * 1e-3), "waves": round(b2 / wave, 2),
                                "sampled_outputs_decrypt_correctly": ok})
            del di, do
        torch.cuda.empty_cache()

    string_ops = None
    if args.string_ops and args.params == "2_2":
        string_ops = bench_string_ops(eng, wl, rank, world, args.exchange)
        try:
            string_ops["multibit_config5"] = bench_multibit_compare(local, rank, world, args.exchange)
        except Exception as e:      # every rank takes the same path; an error must not cost the headline line
            string_ops["multibit_config5"] = {"error": str(e)[:300]}

    if world > 1:
        t = torch.tensor([ms, e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_s = float(t[0]), float(t[1])
        ok = torch.tensor([int(validation["ok"] and e2e_validation["ok"])], device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        validation["all_ranks_ok"] = bool(int(ok[0]))
    if rank == 0:
        peaks, peak_kind = _peaks()
        fp64_peak = eng.probe_fp64_tflops()
        value = B * world * args.steps / (ms * 1e-3)
        e2e = B * world * e2e_steps / e2e_s
        pbs_tflops = B * FLOP / (pbs_ms * 1e-3) / 1e12
        alg_bytes = BSK_BYTES + B * (SMALL_BYTES // 4 + CT_BYTES) + 16 * p.lut_len * 8     # PBS launch: key once, u16 small cts in, big cts out, LUTs
        hbm_alg = (BSK_BYTES + KSK_BYTES + B * (2 * CT_BYTES + 2 * SMALL_BYTES // 4)) / ((pbs_ms + ks_ms) * 1e-3) / 1e9
        cpu = None
        if args.cpu_sample != 0:
            n_cpu = args.cpu_sample if args.cpu_sample > 0 else host_cores() * 320     # about 8-10 s at 30-40 KS-PBS/s per core
            cpu = cpu_reference_rate(wl, n_cpu) + (n_cpu,)
        traffic, traffic_src = None, None
        tf = ROOT / "profiles" / ("r02_pbs_traffic.json" if (ROOT / "profiles" / "r02_pbs_traffic.json").exists() else "r01_pbs_traffic.json")
        if tf.exists() and args.params == "2_2":
            t = json.loads(tf.read_text())
            if t.get("batch") == B:
                traffic, traffic_src = t["dram_bytes"], f"static: dram__bytes_read.sum + dram__bytes_write.sum of one launch at this batch size from the committed ncu capture profiles/{tf.name} (not measured in this run)"
        line = {
            "metric": "batched KS-PBS throughput", "value": value, "unit": "PBS/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{meta['name']} batched KS-PBS ({meta['config'] if args.params != '2_2' else 'configs[1]'})", "batch_per_gpu": B,
                       "luts": 16, "l2_policy": "inputs larger than L2 (cts in+out %.0f MB + keys %.0f MB per step)" % (2 * B * CT_BYTES / 1e6, (BSK_BYTES + KSK_BYTES) / 1e6),
                       "sharding": "ciphertexts partitioned across ranks, keys replicated, no data-path collective",
                       "inputs": "real seeded keys, real encryptions (tile of 256 distinct ciphertexts), 16 lookup tables round-robin"},
            "e2e": {"value": e2e, "unit": "PBS/s", "h2d_bytes_per_step": B * (CT_BYTES + 4), "d2h_bytes_per_step": B * CT_BYTES},
            "gpu_launches": launches,
            "kernels": {"keyswitch_ms": ks_ms, "pbs_ms": pbs_ms},
            "validation": {"device_path": validation, "e2e_path": e2e_validation,
                           "what": "every output ciphertext of the timed batch decrypted (oracle client key) and compared with its LUT value"},
            "roofline": {"bound": "fp64", "kernel": meta["kernel"], "achieved": pbs_tflops, "peak": fp64_peak, "unit": "TFLOP/s",
                         "frac": pbs_tflops / fp64_peak if fp64_peak else None, "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "peak_source": "FP64 FMA microbenchmark run in this process (MEASURED_PEAKS.json has no FP64 figure)",
                         "flop_per_pbs": FLOP,
                         "hbm": {"achieved": hbm_alg, "peak": peaks.get("hbm_gbs"), "unit": "GB/s",
                                 "frac": hbm_alg / peaks["hbm_gbs"] if peaks.get("hbm_gbs") else None, "peak_source": peak_kind}},
            "clocks": _summarise_clocks(samples),
        }
        if batch_sweep:
            line["batch_sweep"] = {"rows": batch_sweep, "note": f"config 2's range; one wave = {(3 if p.grouping_factor else 4) * sms} ciphertexts "
                                   "(whole waves run on the wide kernel, a remainder of at most 2 x SMs on the narrow-level kernel)"}
        if string_ops is not None:
            line["string_ops"] = string_ops
        if args.other_sets and world == 1:
            # breadth, next to the headline: two other classic parameter sets (SURVEY 8f N4), this rank's GPU only
            try:
                line["other_parameter_sets"] = [
                    {k: r[k] for k in ("params", "N", "k", "pbs_level", "batch", "ks_pbs_per_s", "pbs_ms", "pbs_tflops")}
                    for r in param_sweep_rows(args.other_sets.split(","), False, local)]
            except Exception as e:            # never lose the headline over the extra rows
                line["other_parameter_sets"] = {"error": str(e)[:200]}
        if cpu is not None:
            cpu_rate, cpu_cores, cpu_dt, cpu_ok, n_cpu = cpu
            line["cpu_baseline"] = {"value": cpu_rate, "unit": "PBS/s", "cores": cpu_cores, "kind": "port",
                                    "sample": f"{n_cpu} KS-PBS (same keys and ciphertexts as the GPU arm), {cpu_dt:.1f} s", "outputs_decrypt_correctly": cpu_ok}
            if string_ops is not None:
                # the CPU path has no batching effect beyond its cores: a string op costs (its PBS count) / (CPU KS-PBS rate)
                counts = string_ops["pbs_counts"]
                string_ops["cpu_port_ops_per_s_derived"] = {
                    **{k: cpu_rate / float(v) for k, v in counts.items()},
                    "note": "derived: CPU KS-PBS/s of cpu_baseline / PBS count of the unsharded tree (pbs_counts)"}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8192, help="ciphertexts per GPU per step")
    ap.add_argument("--params", default="2_2", choices=["2_2", "multibit"], help="2_2 = PARAM_MESSAGE_2_CARRY_2_KS_PBS (headline); multibit = ..._GROUP_3_KS_PBS")
    ap.add_argument("--string-ops", type=int, default=1, help="also time the FheString operations through the host layer (0 = skip)")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"], help="narrow-end exchange of the sharded string operations")
    ap.add_argument("--batch-sweep", default="4096,16384,65536", help="other batch sizes of config 2, device-timed ('' = skip)")
    ap.add_argument("--param-sweep", default="", help="comma-separated classic sets (e.g. 1_1,3_3,4_4): per-set KS-PBS/s on one GPU + CPU oracle, then exit")
    ap.add_argument("--other-sets", default="1_1,3_3", help="classic sets measured briefly after the headline and reported as other_parameter_sets ('' = skip)")
    ap.add_argument("--cpu-sample", type=int, default=-1, help="KS-PBS evaluated by the CPU baseline leg (-1 = host cores x 320, about 10 s; 0 = skip)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the output ciphertexts of the last timed step to DIR/ks_pbs_out.npy (rank 0 only; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.param_sweep:
        ap.error("--dump-outputs writes the KS-PBS benchmark's outputs; --param-sweep has none to write")
    # stdout carries the one JSON line and nothing else: libraries that write to file descriptor 1 behind Python's back (NCCL's version
    # banner and warnings, OpenMP runtime notices) are sent to stderr; emit() writes the line to the saved descriptor
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if args.param_sweep:
        run_param_sweep(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
