"""
CPU-only: dist.gather_rows, the collective behind the checkpoints of policy-sharded libraries, puts every rank's policy rows
in the single-process order on a world_size-2 gloo group, for even and uneven shards and for the dtypes a library's
training state holds (fp32 rows, int32 Adam step counters).
"""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from deep_successor_features_for_transfer_b200 import dist as sdist
from tests.test_abi_and_dist_cpu import _free_port


def _gather_worker(rank, world, port, full, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        n_total = full[0].shape[0]
        lo, hi = sdist.shard_range(n_total, world, rank)
        ctx = sdist.ShardContext(hi - lo)
        got = [sdist.gather_rows(t[lo:hi], ctx) for t in full]
        into = torch.full_like(full[0], -1.0)
        res = sdist.gather_rows(full[0][lo:hi], ctx, out=into)
        # numpy arrays travel by value: torch tensors would travel as file descriptors this process must outlive
        out.put((rank, [t.numpy() for t in got], into.numpy(), res.data_ptr() == into.data_ptr()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('n_total', [4, 5])
def test_gather_rows_gloo_world2(n_total):
    """4 policies over 2 ranks (2 + 2, one all-gather) and 5 (3 + 2, padded to the larger shard): every rank gets all rows
    in global policy order, with their dtype, bit for bit; `out` is filled in place."""
    g = torch.Generator().manual_seed(3)
    rows = torch.randn(n_total, 37, generator=g)
    rows[1, 5] = float('-0.0')
    steps = torch.randint(0, 1 << 30, (n_total,), generator=g, dtype=torch.int32)
    full = [rows, steps, rows[:, :7].reshape(n_total, 7, 1)]
    ctx = mp.get_context('spawn')
    out = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, full, out)) for r in range(2)]
    for p in procs:
        p.start()
    results = [out.get() for _ in procs]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert sorted(r for r, *_ in results) == [0, 1]
    for rank, got, into, same_buffer in results:
        got, into = [torch.from_numpy(a) for a in got], torch.from_numpy(into)
        for want, have in zip(full, got):
            assert have.dtype == want.dtype and have.shape == want.shape, rank
            assert torch.equal(have.view(torch.int32) if have.dtype == torch.float32 else have,
                               want.view(torch.int32) if want.dtype == torch.float32 else want), rank
        assert torch.equal(into, rows) and same_buffer, rank
