"""Two-GPU parity of the sharded string operations (-m gpu; skipped unless the box has >= 2 GPUs): one process per GPU, real seeded
PARAM_MESSAGE_2_CARRY_2_KS_PBS keys replicated on both, torch.distributed over NCCL for the rendezvous, and BOTH exchange paths --
the engine's own peer-memory kernel over CUDA IPC / NVLink (exchange="peer", the product path) and NCCL (exchange="nccl") -- checked
against clear text after decryption (integer/server_key/radix_parallel/scalar_comparison.rs:147-240 boolean trees,
integer/server_key/comparator.rs:257-279 sign tree) and against each other word for word (the exchanged sums are exact integers)."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, ret):
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{rank}"))
    import fhe_string_bounty_b200 as F
    from fhe_string_bounty_b200 import multi_gpu as MG
    from oracle import oracle as O
    from oracle import radix as R
    from helpers import engine_params
    p = O.params("2_2")
    ck = O.ClientKey(p, 0xB200 + 1)          # same seeds on every rank: keys are replicated
    sk = O.ServerKey(ck, 0xB300 + 1)
    params = engine_params(p)
    eng = F.Engine(params, device=rank)
    eng.upload_ksk(sk.ksk)
    eng.upload_bsk_std(sk.bsk)
    results, raw = [], {}
    for mode in ("peer", "nccl"):
        comm = MG.DeviceComm(eng, exchange=mode)
        comm.min_shard_width = 0                     # shard even these small trees: the test is about the sharded path
        rng = np.random.default_rng(0xB200 + 3)      # same strings on every rank and in both modes
        hay = bytes(rng.integers(ord("a"), ord("z") + 1, size=64).tolist())
        for pat in (hay[37:45], b"zzzzzzzq"):
            h, q = R.encrypt_string(ck, hay), R.encrypt_string(ck, pat)
            out = MG.sharded_contains(comm, params, h, q, len(hay), len(pat))
            results.append((mode, "contains", pat, ck.decrypt_message_and_carry(out), int(pat in hay)))
            out = MG.sharded_find(comm, params, h, q, len(hay), len(pat))
            pos = hay.find(pat)
            results.append((mode, "find", pat, (ck.decrypt_message_and_carry(out[0]), R.decrypt_radix(ck, out[1:])), (int(pos >= 0), max(pos, 0))))
        a = bytes(rng.integers(0x20, 0x7F, size=24).tolist())
        for b in (a, a[:17] + b"~" + a[18:], a[:3] + b" " + a[4:]):
            ea, eb = R.encrypt_string(ck, a), R.encrypt_string(ck, b)
            out = MG.sharded_eq(comm, params, ea, eb, len(a))
            results.append((mode, "eq", b, ck.decrypt_message_and_carry(out), int(a == b)))
            for op, w in (("lt", a < b), ("le", a <= b), ("gt", a > b), ("ge", a >= b)):
                out = MG.sharded_compare(comm, params, op, ea, eb, len(a))
                results.append((mode, op, b, ck.decrypt_message_and_carry(out), int(w)))
        # an ODD number of exchanged rows (1 + 4 index blocks for 241 windows) and alternating operands: a result that is one exchange
        # behind, or assembled on the wrong stream, shows here (bench.py's config 3 shape)
        hay2 = bytes(rng.integers(ord("a"), ord("z") + 1, size=256).tolist())
        pat2 = hay2[201:217]
        h2, q2, q3 = R.encrypt_string(ck, hay2), R.encrypt_string(ck, pat2), R.encrypt_string(ck, b"0123456789ABCDEF")
        for rep in range(2):
            for q, w in ((q2, (1, 201)), (q3, (0, 0)), (q2, (1, 201))):
                out = MG.sharded_find(comm, params, h2, q, 256, 16)
                got = (ck.decrypt_message_and_carry(out[0]), R.decrypt_radix(ck, out[1:]))
                results.append((mode, "find256", rep, got if w[0] else (got[0], 0), w))
                out = MG.sharded_contains(comm, params, h2, q, 256, 16)
                results.append((mode, "contains256", rep, ck.decrypt_message_and_carry(out), w[0]))
        s = b"Hello Zama, how is it going?"
        out = MG.sharded_case(comm, params, "to_lowercase", R.encrypt_string(ck, s), len(s))
        results.append((mode, "lower", s, R.decrypt_string(ck, out), s.lower()))
        # exchange primitives on known rows: exact integer results, identical in both modes
        L = eng.p.big_len
        mine = torch.from_numpy((np.arange(2 * L, dtype=np.uint64).reshape(2, L) * np.uint64(rank + 3)).view(np.int64)).cuda()
        raw[mode] = (comm.to_host(comm.all_reduce(mine.clone())), comm.to_host(comm.all_gather(mine.clone()).reshape(-1, L)))
        comm.close()
    same = np.array_equal(raw["peer"][0], raw["nccl"][0]) and np.array_equal(raw["peer"][1], raw["nccl"][1])
    base = np.arange(2 * L, dtype=np.uint64).reshape(2, L)
    exact = np.array_equal(raw["peer"][0], base * np.uint64(sum(r + 3 for r in range(world))))
    ret[rank] = (results, same, exact)
    eng.close()
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_string_ops_two_gpus_nccl_and_peer():
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    world = 2
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    assert len(ret) == world
    for rank in range(world):
        results, same, exact = ret[rank]
        assert same, "peer-memory exchange and NCCL disagree"
        assert exact, "all-reduce over peer memory is not the exact u64 sum"
        for mode, op, arg, got, want in results:
            assert got == want, (rank, mode, op, arg, got, want)
