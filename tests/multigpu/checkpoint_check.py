"""
Multi-GPU check (torchrun, NCCL): checkpoints of policy-sharded SF libraries.  state_dict() / load_state_dict() of a sharded
library are collectives that save and load the one-GPU format, so

  1. a sharded run saved and restored into fresh sharded objects continues bit for bit (losses, online / target / m / v rows,
     w, g, h, step counters, GPI keys of a probe batch);
  2. the dict is the same on every rank, its rows [lo, hi) are that rank's buffers, and h agrees on every rank before the save;
  3. the dict crosses world sizes: rank 0 loads it into an unsharded library of all N policies (rows bit-equal, K more steps
     within shard_check.py's bounds), a dict of that unsharded library loads back into the shards bit for bit, and with 4 or
     more ranks the world-W dict loads into libraries sharded over the first W/2 ranks (rows and GPI keys bit-equal);
  4. a dict of the wrong policy count raises the same ValueError on every rank and changes nothing; the agents'
     state_dict() / load_state_dict() refuse sharded libraries.

TSF (variant 2, whose shared h is exchanged between ranks) and plain SF (variant 1) libraries, built like shard_check.py.

Arguments: the precision mode (fp32 | bf16 | tf32 | tf32x3) and the shard shape (even | uneven).  Run every mode and shape
with the default peer-memory exchange and again with SFGPI_PEER=0 (the NCCL-collective exchange), and once on 4 ranks:

  python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/multigpu/checkpoint_check.py bf16 even
  SFGPI_PEER=0 python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tests/multigpu/checkpoint_check.py bf16 uneven
  python -m torch.distributed.run --nproc-per-node 4 --master-addr 127.0.0.1 tests/multigpu/checkpoint_check.py fp32 even

Exits non-zero on any failure.  With more ranks than GPUs the ranks share the GPUs over gloo: the collective exchange's code
path, uneven shards only (no peer memory, no fused even-shard exchange).
"""
import io
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
import torch.distributed as dist

from oracle.sf_oracle import OracleSF, synthetic_transitions
from tests import gpu_util as gu
from deep_successor_features_for_transfer_b200.dist import gather_rows, shard_range
from deep_successor_features_for_transfer_b200.sfdqn import SFDQN, ReplayBuffer

precision = sys.argv[1] if len(sys.argv) > 1 else 'fp32'
shape = sys.argv[2] if len(sys.argv) > 2 else 'uneven'
rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
# one GPU per rank over NCCL; with fewer GPUs than ranks the ranks share them over gloo, which runs the NCCL-collective
# exchange's code path (the peer-memory exchange needs NCCL and a GPU per rank)
backend = 'nccl' if world <= torch.cuda.device_count() else 'gloo'
if backend == 'gloo' and shape == 'even':
    sys.exit('checkpoint_check: the fused exchange of even shards needs NCCL (gloo refuses its all-gather shapes): run '
             'even shards with a GPU per rank')
dev = torch.device('cuda', local % torch.cuda.device_count())
torch.cuda.set_device(dev)
dist.init_process_group(backend, **(dict(device_id=dev) if backend == 'nccl' else {}))
S, A, D, B, K = 4, 9, 12, 1000, 3
N = 2 * world + (0 if shape == 'even' else 1)
TOL = 5e-5 if precision == 'fp32' else 5e-3
lo, hi = shard_range(N, world, rank)
half = world // 2 if world >= 4 and world % 2 == 0 else None
half_group = dist.new_group(list(range(half))) if half else None       # (every rank creates it)
fails = []


def check(ok, what):
    if not ok:
        fails.append(f'rank {rank}: {what}')


def oracle(seed):
    g = torch.Generator().manual_seed(seed)
    o = OracleSF(S, A, D, (256, 256), ('relu', 'relu'), tsf_dim=100, beta=1)
    for _ in range(N):
        o.add_random_policy(g)
    return o


O_A, O_B = oracle(5), oracle(6)                                       # the saved run / the runs that load (other weights)
gen = torch.Generator().manual_seed(7)
first, second = ([gu.cuda_tr(synthetic_transitions(B, S, A, D, gen)) for _ in range(K)] for _ in range(2))
spare = gu.cuda_tr(synthetic_transitions(B, S, A, D, gen))
probe = gu.cuda_tr(synthetic_transitions(B, S, A, D, gen))[4]


class Sub:                                                            # oracle view holding policies [lo, hi)
    def __init__(self, o, lo_, hi_):
        self.psi, self.w, self.g, self.h = o.psi[lo_:hi_], o.w[lo_:hi_], o.g[lo_:hi_], o.h


def build(kind, o, lo_, hi_, group=None, shard=True):
    """(SF object, agent, all-task step) over policies [lo_, hi_) of oracle o, sharded over `group` unless shard=False."""
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=hi_ - lo_, gdim=100, beta=1, use_gpi=True)
    if kind == 'tsf':
        sf, ag = gu.build_g3(meta, oracle=Sub(o, lo_, hi_))
        step = lambda tr: ag.update_successor_all(tr, use_gpi=True).clone()
    else:
        sf = gu.build_g2(meta, oracle=Sub(o, lo_, hi_))
        ag = SFDQN(sf, lambda: ReplayBuffer(), 0.9, 500, None)
        step = lambda tr: sf.update_successor_all(tr, use_gpi=True).clone()
    sf._library.set_precision(precision)
    if shard:
        sf._library.enable_sharding(group)
    return sf, ag, step


def rows(lib):
    out = {k: getattr(lib, k).detach()[:lib.n].clone() for k in lib._state_rows()}
    if lib.G is not None:
        out['h'] = lib.h.clone()
    return out


def saved_rows(ls, lo_, hi_):
    """The dict's rows [lo_, hi_) of every per-policy buffer, and h."""
    return {k: (v if k == 'h' else v[lo_:hi_]) for k, v in ls.items() if torch.is_tensor(v)}


def bit_equal(x, y):
    return x.dtype == y.dtype and x.shape == y.shape and torch.equal(x.view(torch.int32), y.view(torch.int32))


def compare_bits(a, b, what):
    for k in a:
        check(bit_equal(a[k], b[k]), f'{what}: {k!r} differs')


def rel(x, y):
    x, y = x.double(), y.double()
    return float((x - y).abs().max() / x.abs().max().clamp_min(1e-30))


def gpi_keys(lib, w_rows, x):
    """GPI keys of states x under every reward vector w_rows[i], all-reduced over the library's group (a collective)."""
    return [torch.cat(lib.gpi(x, w, want_q=False)[1:]) for w in w_rows]


def roundtrip(sd):
    buf = io.BytesIO()
    torch.save(sd, buf)
    buf.seek(0)
    return torch.load(buf, map_location=dev)


def errors_alike(fn, exc, what):
    """fn() raises exc on this rank; the messages of every rank are equal (gathered: no rank is left in a collective)."""
    try:
        fn()
        msg = None
    except exc as e:
        msg = str(e)
    msgs = [None] * world
    dist.all_gather_object(msgs, msg)
    check(msg is not None, f'{what}: no {exc.__name__}')
    check(len(set(msgs)) == 1, f'{what}: the ranks raised different errors {msgs}')
    return msg


def run(kind):
    a, _, step_a = build(kind, O_A, lo, hi)
    lib_a = a._library
    for tr in first:
        step_a(tr)
    if lib_a.G is not None:
        hs = [torch.empty_like(lib_a.h) for _ in range(world)]
        dist.all_gather(hs, lib_a.h)
        check(all(bit_equal(h, hs[0]) for h in hs), f'{kind}: h differs across ranks before the save')
    own = rows(lib_a)
    sd = roundtrip(a.state_dict())
    ls = sd['library']

    # ---- 2. the dict: full-sized, the same on every rank, this rank's rows are its buffers
    check(sd['n_tasks'] == N and ls['online'].shape[0] == N and len(sd['psi']) == N, f'{kind}: the dict is not {N} policies')
    check(all(len(c) == N for c in sd['gpi_counters']) and len(sd['gpi_counters']) == N, f'{kind}: gpi_counters not {N} x {N}')
    check(sd['updates_since_target_updated'] == [K] * N, f"{kind}: updates_since_target_updated {sd['updates_since_target_updated']}")
    compare_bits(own, saved_rows(ls, lo, hi), f'{kind}: dict rows [lo, hi) vs own buffers')
    for k, v in ls.items():
        if torch.is_tensor(v):
            r0 = v.clone()
            dist.broadcast(r0, src=0)
            check(bit_equal(v, r0), f'{kind}: dict {k!r} differs from rank 0')
    for i in (0, N - 1):                                              # psi[i]: the reference layout, views of the dict's rows
        Ws = list(sd['psi'][i]['model'].values())
        check(bit_equal(Ws[0].reshape(-1), ls['online'][i, :Ws[0].numel()]), f'{kind}: psi[{i}] model != online row {i}')
        st = sd['psi'][i]['optim']['state']
        check(int(st[0]['step']) == int(ls['step'][i]), f'{kind}: psi[{i}] optim step')
        check(bit_equal(st[0]['exp_avg'].reshape(-1), ls['m'][i, :Ws[0].numel()]), f'{kind}: psi[{i}] optim exp_avg != m row {i}')
    meta = {k: v for k, v in sd.items() if k not in ('library', 'psi')}
    meta['library'] = {k: v for k, v in ls.items() if not torch.is_tensor(v)}
    metas = [None] * world
    dist.all_gather_object(metas, meta)
    check(all(m == metas[0] for m in metas), f'{kind}: the dict\'s host fields differ across ranks')
    la = [step_a(tr) for tr in second]                                # the uninterrupted run

    # ---- 4. errors: every rank raises alike, before any copy
    b, ag_b, step_b = build(kind, O_B, lo, hi)
    lib_b = b._library
    step_b(spare)                                 # b's exchange state now holds its own w / h, which a load must replace
    before = rows(lib_b)
    bad = dict(ls, **{k: ls[k][:N - 1] for k in lib_b._state_rows()})
    msg = errors_alike(lambda: lib_b.load_state_dict(bad), ValueError, f'{kind}: {N - 1}-policy dict')
    check(msg is not None and f'{N - 1} policies' in msg and f'{N} over {world} ranks' in msg, f'{kind}: message {msg!r}')
    errors_alike(lambda: b.load_state_dict(dict(sd, n_tasks=N + 1)), ValueError, f'{kind}: SF dict of {N + 1} tasks')
    compare_bits(before, rows(lib_b), f'{kind}: a failed load changed the library')
    errors_alike(ag_b.state_dict, NotImplementedError, f'{kind}: agent state_dict')
    errors_alike(lambda: ag_b.load_state_dict({}), NotImplementedError, f'{kind}: agent load_state_dict')

    # ---- 1. same world size, bit for bit
    b.load_state_dict(sd)
    compare_bits(rows(lib_b), saved_rows(ls, lo, hi), f'{kind}: loaded rows vs dict')
    w_rows = ls['w']
    keys_loaded = gpi_keys(lib_b, w_rows, second[0][4])             # what the first resumed step's GPI computes
    lb = [step_b(tr) for tr in second]
    for k, (x, y) in enumerate(zip(la, lb)):
        check(bit_equal(x, y), f'{kind}: losses of resumed step {k} differ')
    compare_bits(rows(lib_a), rows(lib_b), f'{kind}: resumed run vs uninterrupted run')
    check(a.updates_since_target_updated == b.updates_since_target_updated, f'{kind}: updates_since_target_updated')
    for x, y in zip(gpi_keys(lib_a, w_rows, probe), gpi_keys(lib_b, w_rows, probe)):
        check(torch.equal(x, y), f'{kind}: GPI keys of the probe batch differ')

    # ---- 3. across world sizes
    final = a.state_dict()['library']                                 # the sharded continuation, gathered
    la_full = [gather_rows(x, lib_a.shard) for x in la]
    worst, usd = 0.0, None
    if rank == 0:
        u, _, step_u = build(kind, O_B, 0, N, shard=False)
        u.load_state_dict(sd)
        compare_bits(rows(u._library), saved_rows(ls, 0, N), f'{kind}: unsharded load of the world-{world} dict')
        lu = [step_u(tr) for tr in second]
        worst = max(rel(x, y) for x, y in zip(la_full, lu))
        got = rows(u._library)
        for k in ('online', 'w', 'g', 'h'):
            if k in got:
                worst = max(worst, rel(final[k], got[k]))
        check(worst < TOL, f'{kind}: unsharded continuation deviates {worst:.3e} from the sharded one (tol {TOL})')
        buf = io.BytesIO()
        torch.save(u.state_dict(), buf)
        usd = buf.getvalue()
    obj = [usd]
    dist.broadcast_object_list(obj, src=0)
    usd = torch.load(io.BytesIO(obj[0]), map_location=dev)
    b.load_state_dict(usd)
    compare_bits(rows(lib_b), saved_rows(usd['library'], lo, hi), f'{kind}: shard of the unsharded dict')

    bits = None
    if half and rank < half:                                          # W -> W/2: the world-W dict over the first W/2 ranks
        lo2, hi2 = shard_range(N, half, rank)
        c, _, step_c = build(kind, O_B, lo2, hi2, group=half_group)
        c.load_state_dict(sd)
        compare_bits(rows(c._library), saved_rows(ls, lo2, hi2), f'{kind}: world-{half} shard of the world-{world} dict')
        for x, y in zip(keys_loaded, gpi_keys(c._library, w_rows, second[0][4])):
            check(torch.equal(x, y), f'{kind}: GPI keys over {half} ranks differ from those over {world}')
        lc = gather_rows(step_c(second[0]), c._library.shard)
        bits = bit_equal(lc, la_full[0])
        check(rel(la_full[0], lc) < TOL, f'{kind}: first step over {half} ranks deviates {rel(la_full[0], lc):.3e}')
    return worst, bits, lib_a._peer is not None


results = {kind: run(kind) for kind in ('tsf', 'sf')}
torch.cuda.synchronize()
everyone = [None] * world
dist.all_gather_object(everyone, fails)
all_fails = [f for fs in everyone for f in fs]
if rank == 0:                                  # (rank 0 computed both the unsharded deviation and the W/2 first step)
    for f in all_fails:
        print('FAIL', f, flush=True)
    parts = []
    for kind, (worst, bits, _) in results.items():
        parts.append(f'{kind}: unsharded continuation within {worst:.2e}')
        if bits is not None:
            parts[-1] += f', first step over {half} ranks ' + ('bit-equal' if bits else 'within tol')
    peer = all(r[2] for r in results.values())
    print(f'checkpoint_check {precision} {shape} world={world} N={N} backend={backend} peer={peer}: '
          f'{"; ".join(parts)} (tol {TOL}) -> {"FAIL" if all_fails else "OK"}', flush=True)
dist.barrier()
dist.destroy_process_group()
sys.exit(1 if all_fails else 0)
