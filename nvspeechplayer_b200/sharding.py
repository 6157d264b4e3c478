"""Multi-GPU sharding of the batch path: streams are independent (per-stream noise, no shared state), so a job of
`total` streams is cut into contiguous ranges, one per rank, with NO data-path collective (SURVEY.md section 8e).
torch.distributed is only used for the timing barrier and to combine per-rank scalars (max time, sum of samples)."""


def shard_range(total_streams, rank, world):
    """[first, last) of the streams rank `rank` renders: contiguous, sizes differ by at most one."""
    if not (0 <= rank < world):
        raise ValueError("rank %d outside world %d" % (rank, world))
    base, extra = divmod(int(total_streams), int(world))
    first = rank * base + min(rank, extra)
    return first, first + base + (1 if rank < extra else 0)


def weak_shard(streams_per_rank, rank):
    """Weak scaling (bench.py): every rank renders `streams_per_rank` streams; ids are globally unique."""
    first = rank * int(streams_per_rank)
    return first, first + int(streams_per_rank)


def balanced_ranges(ticks_per_stream, shards):
    """first[shards + 1] of contiguous stream ranges whose tick sums are balanced -- the rule speechPlayer_multiBatchSetFramesHost
    applies (api_batch.cu): with upto = running sum of (ticks + 1), shard d starts at the first stream where upto reaches d / shards
    of the total.  tests/test_gpu_multibatch.py holds the library to this function."""
    import numpy as np
    t = np.asarray(ticks_per_stream, dtype=np.uint64) + np.uint64(1)
    upto = np.concatenate([[0], np.cumsum(t, dtype=np.uint64)]).astype(np.uint64)
    n, total = len(t), int(upto[-1])
    first = [0]
    for d in range(1, shards):
        want = total // shards * d + total % shards * d // shards
        f = int(np.searchsorted(upto, np.uint64(want), side="left"))
        first.append(min(max(f, first[-1]), n))
    first.append(n)
    return first


def combine(dist, device, elapsed_ms, samples):
    """(max over ranks of elapsed_ms, sum over ranks of samples) -- the two numbers the benchmark line needs."""
    import torch
    t = torch.tensor([float(elapsed_ms)], dtype=torch.float64, device=device)
    n = torch.tensor([float(samples)], dtype=torch.float64, device=device)
    if dist is not None and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(n, op=dist.ReduceOp.SUM)
    return float(t.item()), float(n.item())
