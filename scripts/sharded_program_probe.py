"""Device time of whole recorded programs run across the ranks with multi_gpu.run_program_sharded, at the world torchrun starts (one
process per GPU; world 1 runs the plain program), with real keys and every result decrypted and checked against Python bytes.

    torchrun --nproc_per_node N scripts/sharded_program_probe.py --out DIR [--reps R] [--log profiles/NAME.log]

Per case it reports the median over R runs of program_last_ms (CUDA events around every level, exchanges included) and of a host clock
around the call that ends in a stream synchronise.  string_contains_packed {256, 16} is timed next to multi_gpu.sharded_contains on the
same inputs.  Rank 0 writes DIR/sharded_program_probe_w<N>.json and appends to the log; the card name and power limit are read in the
same run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]


def card(dev: int) -> dict:
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(dev)], capture_output=True, text=True,
                         timeout=30).stdout.strip()
    name, power, clock = [s.strip() for s in out.split(",")]
    return {"name": name, "power_limit_w": float(power), "max_sm_mhz": float(clock)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--log", default=None)
    ap.add_argument("--only", default=None, help="comma-separated case names")
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("sharded_program_probe.py: no CUDA device")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import fhe_string_bounty_b200 as F
    from fhe_string_bounty_b200 import multi_gpu as MG
    from fhe_string_bounty_b200.host import Program
    from helpers import engine_params
    from oracle import oracle as O, radix as R
    from test_padded_split_replace import digits_for, max_matches, pad, rs_replacen, rs_splitn

    p = O.params("2_2")
    ck = O.ClientKey(p, 0x5EED)
    sk = O.ServerKey(ck, 0x5EEE)
    prm = engine_params(p)
    eng = F.Engine(prm, device=local)
    eng.upload_ksk(sk.ksk)
    eng.upload_bsk_std(sk.bsk)
    comm = MG.DeviceComm(eng)
    dec = ck.decrypt_message_and_carry
    enc = lambda *strings: np.concatenate([R.encrypt_string(ck, pad(s, c)) for s, c in strings])
    s32 = b"ab cd ab ef abab gh ab ijk ab xy"
    s128 = (s32 * 4)[:127] + b"a"

    def check_split(out, s, pat, cap, m_min):
        n = max_matches(cap, m_min) + 1
        nd = digits_for(n)
        want = rs_splitn(s, pat, None)
        parts = [R.decrypt_string(ck, out[nd + 4 * cap * k: nd + 4 * cap * (k + 1)]) for k in range(n)]
        return R.decrypt_radix(ck, out[:nd]) == len(want) and parts == [pad(w, cap) for w in want] + [pad(b"", cap)] * (n - len(want))

    rng = np.random.default_rng(7)
    pairs = [(bytes(rng.integers(97, 100, 8).tolist()), bytes(rng.integers(97, 100, 8).tolist())) for _ in range(4096)]
    hay = bytes(rng.integers(97, 123, 256).tolist())
    pat = hay[201:217]
    cases = {
        "pstring_split {32, 4}": (("pstring_split", (32, 4), None), lambda: enc((s32, 32), (b"ab", 4)),
                                  lambda o: check_split(o, s32, b"ab", 32, 0)),
        "pstring_split {128, 2} clear ab": (("pstring_split", (128, 2), "ab"), lambda: enc((s128, 128)),
                                            lambda o: check_split(o, s128, b"ab", 128, 2)),
        "pstring_replace {32, 4, 4}": (("pstring_replace", (32, 4, 4), None), lambda: enc((s32, 32), (b"ab", 4), (b"XY!", 4)),
                                       lambda o: R.decrypt_string(ck, o) == pad(rs_replacen(s32, b"ab", b"XY!"), 32 + max_matches(32, 0) * 4)),
        "string_eq_many {8, 8, 4096}": (("string_eq_many", (8, 8, 4096), None),
                                        lambda: np.concatenate([R.encrypt_string(ck, x) for a, b in pairs for x in (a, b)]),
                                        lambda o: [dec(r) for r in o] == [int(a == b) for a, b in pairs]),
        "string_contains_packed {256, 16}": (("string_contains_packed", (256, 16), None), lambda: enc((hay, 256), (pat, 16)),
                                             lambda o: dec(o[0]) == 1),
    }
    if args.only:
        cases = {k: v for k, v in cases.items() if k in args.only.split(",")}
    results = {"world": world, "card": card(local), "min_shard_width": comm.min_shard_width, "reps": args.reps, "cases": {}}
    for name, ((op, a, clear), make, ok) in cases.items():
        P = Program(op, a, clear=clear, params=prm)
        x = make()
        xt = torch.from_numpy(np.ascontiguousarray(x).view(np.int64)).pin_memory()
        plan = P.shard_plan(world, comm.min_shard_width)
        dev_ms, wall_ms, good = [], [], True
        for it in range(args.reps + 1):                     # the first run binds the program and creates the exchange: not timed
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            out = comm.to_host(MG.run_program_sharded(comm, P, xt))
            t1 = time.perf_counter()
            good &= bool(ok(out))
            if it:
                dev_ms.append(P.last_ms())
                wall_ms.append((t1 - t0) * 1e3)
        row = {"n_pbs": P.n_pbs, "levels": P.n_levels, "plan": {"split_levels": plan[0], "max_share": plan[1], "rows_received": plan[2]},
               "device_ms_median": float(np.median(dev_ms)), "wall_ms_median": float(np.median(wall_ms)), "device_ms": dev_ms, "correct": good}
        if op == "string_contains_packed":      # the hand-written split of the same operation on the same inputs
            hay_b, pat_b = xt[:4 * 256].numpy().view(np.uint64), xt[4 * 256:].numpy().view(np.uint64)
            sc = []
            for it in range(args.reps + 1):
                if world > 1:
                    dist.barrier()
                t0 = time.perf_counter()
                r = MG.sharded_contains(comm, prm, hay_b, pat_b, 256, 16)
                t1 = time.perf_counter()
                row["correct"] &= dec(r) == 1
                if it:
                    sc.append((t1 - t0) * 1e3)
            row["sharded_contains_wall_ms_median"] = float(np.median(sc))
        results["cases"][name] = row
        P.close()
        if rank == 0:
            print(f"world {world}: {name}: {row['device_ms_median']:.1f} ms device, {row['wall_ms_median']:.1f} ms wall, plan {plan}, "
                  f"correct {row['correct']}" + (f", sharded_contains {row['sharded_contains_wall_ms_median']:.1f} ms wall"
                                                 if "sharded_contains_wall_ms_median" in row else ""), flush=True)
    comm.close()
    eng.close()
    if rank == 0:
        out_dir = Path(args.out)
        out_dir.mkdir(parents=True, exist_ok=True)
        (out_dir / f"sharded_program_probe_w{world}.json").write_text(json.dumps(results, indent=1))
        if args.log:
            with open(args.log, "a") as f:
                c = results["card"]
                f.write(f"# world {world} on {c['name']}, power limit {c['power_limit_w']:.0f} W, max SM clock {c['max_sm_mhz']:.0f} MHz, "
                        f"min_shard_width {results['min_shard_width']}, median of {args.reps} runs\n")
                for name, row in results["cases"].items():
                    f.write(f"{name}: {row['n_pbs']} PBS, plan {row['plan']}, device {row['device_ms_median']:.1f} ms, wall "
                            f"{row['wall_ms_median']:.1f} ms, correct {row['correct']}"
                            + (f", sharded_contains wall {row['sharded_contains_wall_ms_median']:.1f} ms" if "sharded_contains_wall_ms_median" in row else "")
                            + "\n")
    if not all(r["correct"] for r in results["cases"].values()):
        raise SystemExit("sharded_program_probe.py: a decrypted result was wrong")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
