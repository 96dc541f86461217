"""Host logic of bench.py's N > 1 path (no GPU): every rank derives the same LPT split of the one fixed dataset, the
shards are disjoint, cover everything and are balanced to within one sequence."""
import importlib.util
import os

import numpy as np

from conftest import ROOT


def _bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_rank_shards_partition_the_dataset_and_are_balanced():
    bench = _bench()
    seqs = bench.dataset(3000)
    lens = np.array([len(s) for s in seqs])
    for world in (1, 2, 4, 8):
        seen = np.zeros(len(seqs), bool)
        loads = []
        for rank in range(world):
            mine, ids = bench.rank_shard(seqs, rank, world)
            assert [len(s) for s in mine] == [int(lens[k]) for k in ids]
            assert not seen[ids].any(), "a sequence was given to two ranks"
            seen[ids] = True
            loads.append(int(lens[ids].sum()))
        assert seen.all(), "a sequence was given to no rank"
        assert max(loads) - min(loads) <= int(lens.max()), (world, loads)


def test_dump_sample_is_fixed_and_within_64_mb(tmp_path):
    """--dump-outputs: the same transcripts every run, and at most 64 MB of float32 even if all were 5,000 nt."""
    bench = _bench()
    ids = bench.dump_sample(100_000)
    assert np.array_equal(ids, bench.dump_sample(100_000))
    assert len(np.unique(ids)) == len(ids) == bench.DUMP_TRANSCRIPTS and ids.min() >= 0 and ids.max() < 100_000
    assert len(ids) * 2 * 5000 * 4 <= 64 << 20
    assert np.array_equal(bench.dump_sample(10), np.arange(10))
    outputs = {int(g): (np.full(int(g) % 7, g, np.float32), np.full(int(g) % 7, -g, np.float32)) for g in ids}
    bench.write_dump(str(tmp_path), ids, outputs)
    acc, cond = np.load(tmp_path / "acc.npy"), np.load(tmp_path / "cond.npy")
    assert acc.dtype == cond.dtype == np.float32
    assert np.array_equal(acc, np.concatenate([outputs[int(g)][0] for g in ids])) and np.array_equal(cond, -acc)
    assert np.array_equal(np.load(tmp_path / "transcript_index.npy"), ids.astype(np.float64))
    assert np.array_equal(np.load(tmp_path / "lengths.npy"), (ids % 7).astype(np.float64))


def test_split_matches_the_cpp_partitioner_rule():
    """priblast_b200.distributed.lpt_shard = csrc/host/db_format.cpp lpt_partition: longest first onto the least loaded
    part, ties to the lowest part index."""
    from priblast_b200.distributed import lpt_shard
    lens = [900, 900, 500, 400, 400, 300, 100]
    parts = lpt_shard(lens, 3)
    assert [[int(k) for k in p] for p in parts] == [[0, 4], [1, 5], [2, 3, 6]]
