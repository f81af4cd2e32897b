# -*- coding: UTF-8 -*-
"""
Policy sharding across GPUs (one process per GPU, torch.distributed over NCCL/NVLink).

The ensemble shards naturally over policies j: GPU g owns psi_j, psi^-_j, w_j, g_j and their Adam state for j in
[g*N/G, (g+1)*N/G); the replay batch is replicated.  The only coupling is GPI's max over j, which is exchanged as packed
(value, index) int64 keys with a MAX all-reduce (the keys are built so that SIGNED int64 max == (max q, then smallest index),
i.e. torch.argmax's first-index rule -- see include/sfgpi.h).  Backward and Adam are rank-local; TSF's shared h keeps one Adam
state per policy-optimizer, so ranks exchange only their h deltas (a SUM all-reduce of D*G+D floats).

The host-side mirrors `pack_keys` / `unpack_keys` restate the device packing in torch ops; the CPU (gloo) tests use them.
"""
import torch
import torch.distributed as dist


def shard_range(n_total, world, rank):
    """Contiguous, as-even-as-possible policy range of `rank`; the first n_total % world ranks own one extra policy."""
    base, rem = divmod(n_total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def pack_keys(values, indices):
    """torch mirror of csrc/common.cuh::pack_key: fp32 values [*], integer indices [*] -> int64 keys.  A NaN value packs as
    -inf, as the device epilogues treat it: never selected (a packed NaN would order above +inf)."""
    v = values.float()
    v = (torch.where(v.isnan(), float('-inf'), v) + 0.0).contiguous()
    bits = v.view(torch.int32).to(torch.int64)
    ordered = torch.where(bits >= 0, bits, bits ^ 0x7FFFFFFF)
    low = (0xFFFFFFFF - indices.to(torch.int64)) & 0xFFFFFFFF
    return (ordered << 32) | low


def unpack_keys(keys):
    """int64 keys -> (fp32 values, int64 indices)."""
    low = keys & 0xFFFFFFFF
    idx = 0xFFFFFFFF - low
    ordered = keys >> 32                                            # arithmetic shift keeps the sign
    bits = torch.where(ordered >= 0, ordered, ordered ^ 0x7FFFFFFF).to(torch.int32)
    return bits.view(torch.float32), idx


def gpi_keys_from_q(q, task_base=0):
    """q [B, n_local, A] -> (key_action [B], key_task [B]) for this rank's shard (host mirror of the fused epilogue)."""
    B, n, A = q.shape
    a_idx = torch.arange(A, device=q.device).view(1, 1, A).expand(B, n, A)
    j_idx = (task_base + torch.arange(n, device=q.device)).view(1, n, 1).expand(B, n, A)
    ka = pack_keys(q, a_idx).reshape(B, -1).max(dim=1).values
    kt = pack_keys(q, j_idx).reshape(B, -1).max(dim=1).values
    return ka, kt


def allreduce_max_keys(keys, group=None):
    """In-place MAX all-reduce of packed keys (int64): NCCL ncclMax over NVLink on GPUs, gloo on CPU."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(keys, op=dist.ReduceOp.MAX, group=group)
    return keys


def gather_rows(t, shard, out=None):
    """
    Collective over shard.group: every rank's rows t [n_local, ...] -> [n_total, ...] in global policy order (rank r's rows
    at [lo_r, lo_r + counts[r])), into `out` when given.  Uneven counts travel padded to the largest shard, so one
    all-gather serves every backend (gloo has no uneven all-gather).
    """
    t = t.contiguous()
    if out is None:
        out = t.new_empty((shard.n_total,) + tuple(t.shape[1:]))
    if shard.uniform:
        dist.all_gather_into_tensor(out, t, group=shard.group)
        return out
    m = max(shard.counts)
    pad = t.new_zeros((m,) + tuple(t.shape[1:]))
    pad[:t.shape[0]] = t
    allp = t.new_empty((shard.world * m,) + tuple(t.shape[1:]))
    dist.all_gather_into_tensor(allp, pad, group=shard.group)
    torch.cat([allp[r * m:r * m + c] for r, c in enumerate(shard.counts)], out=out)
    return out


class ShardContext:
    """Rank-local view of a policy-sharded library: which global policy indices live here."""

    def __init__(self, n_local, group=None):
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        counts = torch.tensor([n_local], dtype=torch.int64)
        if self.world > 1:
            dev = torch.device('cuda', torch.cuda.current_device()) if dist.get_backend(group) == 'nccl' else torch.device('cpu')
            allc = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(self.world)]
            dist.all_gather(allc, counts.to(dev), group=group)
            self.counts = [int(c) for c in allc]
        else:
            self.counts = [n_local]
        self.n_total = sum(self.counts)
        self.lo = sum(self.counts[:self.rank])
        self.uniform = len(set(self.counts)) == 1
