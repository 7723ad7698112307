"""CPU: the host side of summarisation -- Summary.to_lists, and gather_summaries under gloo with world size 2 (uneven shards)."""
import os

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mmbidaf_b200.decode import get_generated_indices, greedy_search
from mmbidaf_b200.summarize import Summary, gather_summaries
from mmbidaf_b200.trainer import shard_range


def _summary_of(dist_: torch.Tensor, lengths):
    """A Summary as MMBiDAF.summarize lays it out, from decode.greedy_search (the rule the device selection reproduces)."""
    B, S, _ = dist_.shape
    picks = [greedy_search(dist_[b], lengths[b]) for b in range(B)]
    idx = torch.full((B, S), -1, dtype=torch.int32)
    for b, ks in enumerate(picks):
        idx[b, :len(ks)] = torch.tensor(ks, dtype=torch.int32)
    return Summary(dist_, None, idx, torch.tensor([len(ks) for ks in picks], dtype=torch.int32))


def _case(seed, B=7, S=9, M=14):
    g = torch.Generator().manual_seed(seed)
    lengths = torch.randint(2, M + 1, (B,), generator=g).tolist()
    return torch.rand(B, S, M, generator=g), lengths


def test_to_lists_equals_get_generated_indices():
    for seed in range(5):
        d, lengths = _case(seed)
        assert _summary_of(d, lengths).to_lists() == get_generated_indices(d, lengths)


def test_to_lists_of_empty_and_full_summaries():
    s = Summary(torch.zeros(2, 3, 4), None, torch.tensor([[-1, -1, -1], [3, 0, 3]], dtype=torch.int32),
                torch.tensor([0, 3], dtype=torch.int32))
    assert s.to_lists() == [[], [3, 0, 3]]


def _worker(rank, world, port, n, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    d, lengths = _case(11, B=n)
    rows = list(shard_range(n, rank, world))
    shard = _summary_of(d[rows], [lengths[i] for i in rows])
    out[rank] = gather_summaries(shard)
    dist.destroy_process_group()


def test_gather_summaries_two_gloo_ranks_uneven_shards():
    world = 2
    for n in (5, 2, 8):                                    # 3 + 2, 1 + 1, 4 + 4 videos
        port = 29500 + (os.getpid() + n) % 2000
        with mp.Manager() as mgr:
            out = mgr.dict()
            mp.spawn(_worker, args=(world, port, n, out), nprocs=world, join=True)
            got = {r: out[r] for r in range(world)}
        d, lengths = _case(11, B=n)
        assert got[1] is None
        assert got[0] == get_generated_indices(d, lengths)


def test_gather_summaries_without_a_process_group_is_to_lists():
    d, lengths = _case(3)
    s = _summary_of(d, lengths)
    assert gather_summaries(s) == s.to_lists()
