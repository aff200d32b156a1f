"""The shard plan of tfhe_b200_program_run_sharded on the CPU: which levels are split across the ranks and which PBS jobs each rank runs.

The executor takes every share from tfhe_b200_program_level_share, so these tests check the shares the GPU runs, for the programs of the
multi-GPU issue's table and one program per op family of tests/test_gpu_exact_programs.py."""
import pytest

from fhe_string_bounty_b200.host import Program
from fhe_string_bounty_b200.multi_gpu import shard_range
from test_gpu_exact_programs import PROGRAMS_2_2

WIDE_PROGRAMS = [
    ("pstring_split", (32, 4), None), ("pstring_split", (128, 2), "ab"), ("pstring_replace", (32, 4, 4), None),
    ("pstring_replace", (128, 2, 2), "ab"), ("pstring_contains", (128, 16), None), ("string_eq_ignore_case", (1024, 1024), None),
    ("string_rfind", (256, 16), None), ("string_eq_many", (8, 8, 512), None),
]
ALL = WIDE_PROGRAMS + PROGRAMS_2_2
SMS = 148


def _ids(specs):
    return [f"{op}{list(args)}" + (f"-{clear}" if clear else "") for op, args, clear in specs]


@pytest.fixture(scope="module", params=ALL, ids=_ids(ALL))
def prog(request):
    op, args, clear = request.param
    return Program(op, args, clear=clear)


def _level_widths(P):
    ir = P.ir()
    return [int(ir.level_pbs_off[i + 1] - ir.level_pbs_off[i]) for i in range(P.n_levels)]


@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("min_w", ["0", "sms", "above"])
def test_shares_partition_every_level(prog, world, min_w):
    widths = _level_widths(prog)
    m = {"0": 0, "sms": SMS, "above": max(widths, default=0)}[min_w]
    n_split, max_share, rows = 0, 0, 0
    for lv, w in enumerate(widths):
        shares = [prog.level_share(lv, r, world, m) for r in range(world)]
        split = {s[2] for s in shares}
        assert len(split) == 1, f"level {lv}: the ranks disagree on whether it is split"
        split = split.pop()
        assert split == (world > 1 and w > m), f"level {lv} of width {w}: split={split} at world {world}, min_shard_width {m}"
        if not split:
            assert all(s[:2] == (0, w) for s in shares), f"replicated level {lv}: every rank runs [0, {w})"
            continue
        owner = [0] * w
        for r, (lo, hi, _) in enumerate(shares):
            assert (lo, hi) == shard_range(w, r, world), f"level {lv}, rank {r}"
            for j in range(lo, hi):
                owner[j] += 1
        assert owner == [1] * w, f"level {lv}: a PBS job outside every share or in two of them"
        n_split += 1
        max_share = max(max_share, max(hi - lo for lo, hi, _ in shares))
        rows += w
    assert prog.shard_plan(world, m) == (n_split, max_share, rows)
    if world == 1 or min_w == "above":
        assert n_split == 0


def test_widest_share_sizes_the_exchange():
    """string_eq_many {8, 8, 4096} at world 2: a share of 65 536 rows, 2.15 GB of double-buffered send area per rank at 2_2"""
    P = Program("string_eq_many", (8, 8, 4096))
    assert max(P.level_widths) == 131072
    n_split, max_share, _ = P.shard_plan(2, SMS)
    assert max_share == 65536 and n_split >= 1
    assert 2 * max_share * P.p.big_len * 8 == 2_148_532_224


def test_plan_rejects_bad_arguments():
    from fhe_string_bounty_b200._native import NativeError
    P = Program("string_eq", (4, 4))
    with pytest.raises(NativeError, match="world"):
        P.shard_plan(0, 0)
    with pytest.raises(NativeError, match="rank < world"):
        P.level_share(0, 2, 2, 0)
    with pytest.raises(NativeError, match="no level"):
        P.level_share(P.n_levels, 0, 2, 0)
