"""
-m gpu: the GPI selection rule on exact ties, signed zeros and non-finite q, in every precision mode and on every device path
that builds or reads packed keys.

The rule (include/sfgpi.h, DESIGN.md "Packed keys"): the largest q and, among the cells holding it, the smallest index, with
-0 == +0 (torch.argmax's first-index rule); a NaN is never selected; a (state, reward vector) whose cells are all NaN or -inf
decodes to index 0 (action 0, task task_base).  tests/gpu_util.py::gpi_rule is its float64 statement, and every index below is
compared with it exactly: no tolerance, so a kernel that broke a tie toward the larger index, packed an index wrongly or left a
key unwritten fails.

Exact q in every mode: the psi nets pass the state through the hidden layers unchanged (identity rows, ReLU on states >= 0)
and the output layer reads it with small integer weights, so psi(x) = Wo x + bo and q = psi . w are small integers wherever bf16,
tf32 and fp32 round or sum them, in any order (the folded GPI weights too).  The tables of fixed q (ties, +-0, +-inf, NaN) set
Wo = 0 and choose bo: psi is then bo for every state, and q = bo[a, 0] under w = e_0.

Launch sizes as in tests/test_gpu_architectures.py: 'chain' (N = 3, B = 333) and 'pair' (N = 2, B = 75 * 128 + 7).  A * D = 288
> 256: the fp32 GPI epilogue runs in two column chunks (8 actions, then 1).
"""
import pytest
import torch

from deep_successor_features_for_transfer_b200 import _lib, dist as sdist, workloads as wl
from deep_successor_features_for_transfer_b200.library import _stream
from tests import gpu_util as gu

pytestmark = pytest.mark.gpu

S, A, D, H = 4, 9, 32, 256
MODES = ('fp32', 'bf16', 'tf32', 'tf32x3')
BATCHES = {'chain': (3, 333), 'pair': (2, 75 * 128 + 7)}
SEED = 4321
INF, NAN = float('inf'), float('nan')


def build(precision, N, warm_start=False):
    """DeepSF with the headline hidden layers; warm_start: policies 1.. are copies of policy 0 (add_training_task(source=0))."""
    from deep_successor_features_for_transfer_b200.sfdqn import DeepSF
    sf = DeepSF(pytorch_model_handle=wl.model_lambda([H, H], ['relu', 'relu']), target_update_ev=1000,
                hyperparameters=dict(wl.HYPER, precision=precision))
    sf.reset()
    for k in range(N):
        with wl.seeded_policy_init(SEED + k):
            sf.add_training_task(wl.ShapeTask(S, A, D, k), source=0 if warm_start and k > 0 else None)
    return sf


def load_exact(sf, p, Wo, bo, w):
    """Policy p (online and target) computes psi(x) = Wo x + bo exactly: Wo [A*D, S], bo [A*D]; fit_w[p] = w."""
    eye = torch.zeros(H, S)
    eye[:S, :S] = torch.eye(S)
    W1 = torch.zeros(H, H)
    W1[:S, :S] = torch.eye(S)
    Wout = torch.zeros(A * D, H)
    Wout[:, :S] = Wo
    n_hidden = len(gu.linears(sf.psi[p][0][0].net)) - 2
    gu.load_policy(sf, p, [(eye, torch.zeros(H))] + [(W1, torch.zeros(H))] * n_hidden + [(Wout, bo.float())], w.float())


def exact_states(B, gen):
    return torch.randint(0, 3, (B, S), generator=gen).float()


def psi64(Wo, bo, x):
    return (x.double() @ Wo.double().t() + bo.double()).view(-1, A, D)


def q64(nets, x, w):
    """q [B, N, A] in float64 of the exact nets [(Wo, bo)] under reward vector w [D]."""
    return torch.stack([psi64(Wo, bo, x) @ w.double() for Wo, bo in nets], dim=1)


def random_nets(N, gen):
    """Tie-rich exact nets: sparse {-1, 0, 1} readout of the state, biases in {0, 1}."""
    nets = []
    for _ in range(N):
        Wo = torch.randint(-1, 2, (A * D, S), generator=gen).float() * (torch.rand(A * D, S, generator=gen) < 0.15)
        nets.append((Wo, torch.randint(0, 2, (A * D,), generator=gen).float()))
    return nets


# ---- the fixed q tables ------------------------------------------------------------------------------------------------------
def tables(N, gen):
    """name -> q [N, A] (float32 values; NaN of both signs).  Every case is read under w = e_0."""
    t = {}
    q = torch.zeros(N, A)
    for p in range(N):
        q[p] = torch.arange(A) % 3 + p
        q[p, [3, 6]] = 5 + p                         # policy p's maximum at actions 3 and 6; policy N-1 the best
    t['actions'] = q
    q = -(torch.arange(A) - 4.0).abs().repeat(N, 1)
    q[:, 7] = 0.0
    t['policies'] = q                                # every policy ties at actions 4 and 7
    q = torch.zeros(N, A)
    q[1:, 3:] = 2.0
    t['both'] = q                                    # policies 1.. tie at actions 3.. : action 3, task 1
    q = torch.randint(-3, 2, (N, A), generator=gen).float()
    q[0, 6], q[1, 2] = 7.0, 7.0
    t['divergent'] = q                               # task 0's best is action 6, the key's action is 2
    q = torch.where(torch.rand(N, A, generator=gen) < 0.5, 0.0, -0.0)
    t['signed_zero'] = q
    q = torch.randint(-3, 2, (N, A), generator=gen).float()
    q[N - 1, 4], q[0, 5], q[N - 1, 8] = INF, INF, INF
    t['pos_inf'] = q
    t['neg_inf'] = torch.full((N, A), -INF)
    t['nan'] = torch.full((N, A), NAN)
    q = torch.full((N, A), NAN)
    q[:, 1::2] = (torch.tensor(NAN).view(torch.int32) | -2 ** 31).view(torch.float32)      # the negative NaN
    q[0, 3], q[1, 3] = -INF, -INF
    t['nan_neg_inf'] = q
    q = torch.randint(-3, 2, (N, A), generator=gen).float()
    q[:, 0], q[0, 8] = NAN, NAN
    q[N - 1, 5], q[0, 7] = 3.0, 3.0
    q[1, 2] = -INF
    t['nan_beside_max'] = q                          # NaN at action 0 of every policy: the max is 3 at (N-1, 5) and (0, 7)
    return t


def table_net(q):
    """Wo = 0, bo[a*D] = q[a]: psi = e_0 * q for every state."""
    bo = torch.zeros(A, D)
    bo[:, 0] = q
    return torch.zeros(A * D, S), bo.reshape(-1)


# ---- the device paths --------------------------------------------------------------------------------------------------------
def multi_keys(lib, x, W, w_diag=False, lo=0, n_pol=None):
    """Keys of a fused forward scoring n_w reward vectors W [n_w, D] at once (w_diag: policy p under W[p] only)."""
    n_pol = lib.n - lo if n_pol is None else n_pol
    B = x.shape[0]
    ka = torch.empty(W.shape[0], B, dtype=torch.int64, device='cuda')
    kt = torch.empty_like(ka)
    _lib.call('sfgpi_keys_fill', ka.data_ptr(), ka.numel(), _stream())
    _lib.call('sfgpi_keys_fill', kt.data_ptr(), kt.numel(), _stream())
    wd = W.float().cuda().contiguous()
    a = lib._fwd_args(lib.online, lo, n_pol, x)
    a.w, a.n_w, a.w_diag, a.task_base = wd.data_ptr(), W.shape[0], int(w_diag), lo
    a.key_action, a.key_task = ka.data_ptr(), kt.data_ptr()
    lib._forward(a, 'online')
    act, val = lib.decode_keys(ka, want_value=True)
    return act.cpu(), val.cpu(), lib.decode_keys(kt).cpu()


def check_keys(msg, q, act, task, val=None, task_base=0):
    """act / task / val [B] of one reward vector against the rule on the exact q [B, N, A]."""
    B, N, _ = q.shape
    a_ref, m = gu.gpi_rule(q.reshape(B, -1), torch.arange(A).repeat(N))
    t_ref, _ = gu.gpi_rule(q.reshape(B, -1), (task_base + torch.arange(N)).repeat_interleave(A))
    assert ((act >= 0) & (act < A)).all() and ((task >= task_base) & (task < task_base + N)).all(), (msg, 'index out of range')
    bad = (act != a_ref).nonzero().reshape(-1)
    assert len(bad) == 0, (msg, 'action', len(bad), int(bad[0]), int(act[bad[0]]), int(a_ref[bad[0]]), q[bad[0]])
    bad = (task != t_ref).nonzero().reshape(-1)
    assert len(bad) == 0, (msg, 'task', len(bad), int(bad[0]), int(task[bad[0]]), int(t_ref[bad[0]]), q[bad[0]])
    if val is not None:
        assert torch.equal(val.double(), m), (msg, 'key value')


def target_q_action(psi1, w, omegas):
    """sfgpi_target_q on one state's psi [N][A][D] -> (q [A], action)."""
    N = psi1.shape[0]
    q = torch.empty(A, device='cuda')
    act = torch.empty(1, dtype=torch.int64, device='cuda')
    om, wv, ps = omegas.float().cuda(), w.float().cuda(), psi1.contiguous()
    _lib.call('sfgpi_target_q', ps.data_ptr(), N, A, D, om.data_ptr(), wv.data_ptr(), q.data_ptr(), act.data_ptr(), _stream())
    return q.cpu(), int(act.cpu())


def check_paths(msg, sf, x, w, q, n_target_states=6):
    """One reward vector w over every policy, through every path that selects from q: the fused GPI (keys, q_out), gpi_select,
    gpi_from_psi on the materialised psi, target_q on a mixture of the policies and the host mirror dist.gpi_keys_from_q."""
    lib = sf._library
    N, B = lib.n, x.shape[0]
    xc = x.cuda()
    qd, ka, kt = lib.gpi(xc, w)
    act, val = lib.decode_keys(ka, want_value=True)
    check_keys(msg + ' gpi()', q, act.cpu(), lib.decode_keys(kt).cpu(), val.cpu())
    torch.testing.assert_close(qd.cpu().double(), q, rtol=0, atol=0, equal_nan=True, msg=f'{msg}: gpi() q')
    sel = lib.gpi_select(xc, w).cpu()
    check_keys(msg + ' gpi_select', q, sel[0], sel[1])
    psi = lib.forward_psi(xc)
    _, ka, kt = lib.gpi_from_psi(psi, w)
    act, val = lib.decode_keys(ka, want_value=True)
    check_keys(msg + ' gpi_from_psi', q, act.cpu(), lib.decode_keys(kt).cpu(), val.cpu())
    ka, kt = sdist.gpi_keys_from_q(q.float())
    (va, ia), (_, it) = sdist.unpack_keys(ka), sdist.unpack_keys(kt)
    check_keys(msg + ' dist.gpi_keys_from_q', q, ia, it, va)
    # target_q: q[a] = w . sum_j (omega_j / sum omega) psi_j[a]; omega a power of two in total, so every mixture is exact
    omegas = torch.ones(N)
    omegas[-1] = 1 << (N - 1).bit_length()
    omegas[-1] -= N - 1
    mix = omegas.double() / omegas.sum()
    for b in torch.linspace(0, B - 1, n_target_states).long().tolist():
        qt, at = target_q_action(psi[b], w.reshape(-1), omegas)
        qr = torch.einsum('j,jad->ad', mix, psi[b].cpu().double()) @ w.reshape(-1).cpu().double()
        ar, _ = gu.gpi_rule(qr, torch.arange(A))
        assert at == int(ar), (msg, 'target_q', b, at, int(ar), qr)


def fit_w(sf, p):
    return sf.fit_w[p].weight.detach().reshape(-1)


# ---- the tests -----------------------------------------------------------------------------------------------------------
CASES = [pytest.param(prec, batch, id=f'{prec}-{batch}') for prec in MODES for batch in BATCHES]


@pytest.mark.parametrize('precision,batch', CASES)
def test_fixed_tables(precision, batch):
    """Ties across actions, across policies, both, divergent best actions, +-0, +-inf, all -inf, all NaN, NaN beside a finite
    maximum: every path, and the same tables per policy under w_diag (one reward vector per policy slot)."""
    N, B = BATCHES[batch]
    gen = torch.Generator().manual_seed(11)
    sf = build(precision, N)
    x = exact_states(B, gen)
    e0 = torch.zeros(D)
    e0[0] = 1.0
    for name, t in tables(N, gen).items():
        nets = [table_net(t[p]) for p in range(N)]
        for p, (Wo, bo) in enumerate(nets):
            load_exact(sf, p, Wo, bo, e0)
        q = q64(nets, x, e0)
        assert torch.equal(q[0].isnan(), t.isnan()) and torch.equal(q[0][~t.isnan()], t[~t.isnan()].double())
        check_paths(f'{precision} {batch} {name}', sf, x, fit_w(sf, 0), q)
        act, val, task = multi_keys(sf._library, x.cuda(), e0.repeat(N, 1), w_diag=True)
        for p in range(N):
            check_keys(f'{precision} {batch} {name} w_diag slot {p}', q[:, p:p + 1], act[p], task[p], val[p], task_base=p)


@pytest.mark.parametrize('precision,batch', CASES)
@pytest.mark.parametrize('n_w', [1, 13, 32])
def test_state_dependent_exact_tables(precision, batch, n_w):
    """Tie-rich integer q that varies per state, for 1, 13 (blocked column order, a padded block) and 32 reward vectors in one
    launch; bf16 also through the ping-pong pair kernel (forward_chain 0, with the 32-column-window scan for 32 vectors) and the
    layer-pipelined kernel (forward_chain 2)."""
    N, B = BATCHES[batch]
    gen = torch.Generator().manual_seed(100 + n_w)
    sf = build(precision, N)
    lib = sf._library
    nets = random_nets(N, gen)
    W = torch.randint(-1, 2, (n_w, D), generator=gen).float()
    for p, (Wo, bo) in enumerate(nets):
        load_exact(sf, p, Wo, bo, W[0])
    x = exact_states(B, gen)
    qs = [q64(nets, x, W[k]) for k in range(n_w)]
    ties = sum(int(((qk.reshape(B, -1) == qk.reshape(B, -1).max(dim=1, keepdim=True).values).sum(dim=1) > 1).sum()) for qk in qs)
    assert ties > B * n_w // 8, "the tables should tie at the maximum on many states"
    msg = f'{precision} {batch} n_w={n_w}'
    if n_w == 1:
        check_paths(msg, sf, x, W[0], qs[0])
    runs = [(None, None)]
    if precision == 'bf16':
        runs += [(0, 8 if n_w == 32 else None), (2, None)]
    for chain, wide_min in runs:
        olds = []
        if chain is not None:
            olds.append(('forward_chain', _lib.lib().sfgpi_set_option(b'forward_chain', chain)))
        if wide_min is not None:
            olds.append(('gpi_wide_min', _lib.lib().sfgpi_set_option(b'gpi_wide_min', wide_min)))
        try:
            act, val, task = multi_keys(lib, x.cuda(), W)
            wd = W[:N] if n_w >= N else W[0].repeat(N, 1)
            dact, dval, dtask = multi_keys(lib, x.cuda(), wd, w_diag=True)
        finally:
            for name, old in olds:
                _lib.lib().sfgpi_set_option(name.encode(), old)
        for k in range(n_w):
            check_keys(f'{msg} chain={chain} vector {k}', qs[k], act[k], task[k], val[k])
        for p in range(N):
            qp = q64(nets[p:p + 1], x, wd[p])
            check_keys(f'{msg} chain={chain} w_diag slot {p}', qp, dact[p], dtask[p], dval[p], task_base=p)


@pytest.mark.parametrize('precision,batch', CASES)
def test_warm_start_and_duplicated_actions(precision, batch):
    """State-dependent ties of trained-looking nets: policies warm-started as copies of policy 0 (add_training_task(source=0))
    tie on every state, bit for bit, and the task key takes policy 0; an action whose output rows are copied into a larger
    action ties with it on every state, and the smaller one is selected wherever they are the maximum.  greedy_action and the
    GPI counters follow the same rule."""
    N, B = BATCHES[batch]
    gen = torch.Generator().manual_seed(7)
    sf = build(precision, N, warm_start=True)
    lib = sf._library
    msg = f'{precision} {batch}'
    x = torch.randn(B, S, generator=gen).cuda()
    w = fit_w(sf, 0)
    q, ka, kt = lib.gpi(x, w)
    q = q.cpu()
    for p in range(1, N):
        assert torch.equal(q[:, p], q[:, 0]), (msg, 'a warm-started policy computes other q than its source', p)
    act, val = lib.decode_keys(ka, want_value=True)
    check_keys(msg + ' warm start', q.double(), act.cpu(), lib.decode_keys(kt).cpu(), val.cpu())
    assert int(lib.decode_keys(kt).max()) == 0
    one = [lib.decode_keys(lib.gpi(x, w, lo=p, n_pol=1, want_q=False, task_base=0)[1], want_value=True) for p in range(N)]
    for p in range(1, N):
        assert torch.equal(one[p][0], one[0][0]) and torch.equal(one[p][1], one[0][1]), (msg, 'per-policy keys differ', p)

    # agent level: c = first maximal task, a = first maximal action of row c
    for b in range(4):
        counts = sf.gpi_counters[0].copy()
        a = int(sf.greedy_action(x[b:b + 1], 0))
        qb = lib.gpi(x[b:b + 1], w)[0][0].cpu().double()              # the q of the same launch size
        c_ref = int(gu.gpi_rule(qb.max(dim=1).values, torch.arange(N))[0])
        a_ref = int(gu.gpi_rule(qb[c_ref], torch.arange(A))[0])
        assert (a, sf.gpi_counters[0][c_ref] - counts[c_ref], int(sf.gpi_counters[0].sum() - counts.sum())) == (a_ref, 1, 1), (msg, b)

    # action 2 copied into 6 and action 0 into 8, with action 2 lifted so that it is the maximum on most states
    for p in range(N):
        layers = gu.psi_params(sf, p)
        Wo, bo = layers[-1][0].clone(), layers[-1][1].clone()
        bo[2 * D:3 * D] += 3.0 * w.cpu() / float(w.dot(w))
        for a_src, a_dup in ((2, 6), (0, 8)):
            Wo[a_dup * D:(a_dup + 1) * D], bo[a_dup * D:(a_dup + 1) * D] = Wo[a_src * D:(a_src + 1) * D], bo[a_src * D:(a_src + 1) * D]
        gu.load_policy(sf, p, layers[:-1] + [(Wo, bo)], w.cpu())
    q, ka, kt = lib.gpi(x, w)
    q = q.cpu()
    assert torch.equal(q[..., 6], q[..., 2]) and torch.equal(q[..., 8], q[..., 0]), (msg, 'duplicated rows compute other q')
    act, val = lib.decode_keys(ka, want_value=True)
    check_keys(msg + ' duplicated actions', q.double(), act.cpu(), lib.decode_keys(kt).cpu(), val.cpu())
    assert int((act == 2).sum()) > B // 2 and int((act == 6).sum()) == 0 and int((act == 8).sum()) == 0


def td_reference(nets, tr, i, w_i, next_a):
    """(l1, l2) of the G2 step of policy i (sfdqn.py:330-345) with next actions next_a [B], in float64."""
    states, actions, rs, phis, next_states, gammas = (t.double() for t in tr)
    B = states.shape[0]
    idx = torch.arange(B)
    Wo, bo = nets[i]
    cur = psi64(Wo, bo, states)[idx, actions.long()]
    nxt = psi64(Wo, bo, next_states)[idx, next_a]
    l1 = ((cur - phis - gammas[:, None] * nxt) ** 2).sum() / (B * A * D)
    l2 = ((phis @ w_i.double() - rs.reshape(-1)) ** 2).mean()
    return float(l1), float(l2)


@pytest.mark.parametrize('precision,batch', CASES)
@pytest.mark.parametrize('policy', ['single', 'all'])
def test_train_step_takes_the_rule_action(precision, batch, policy):
    """The fused train step's a* on tie tables whose tied actions have different psi- rows (psi_a = e_0, psi_a' = e_1 under
    w = e_0 + e_1, in every policy at other actions): which one it took shows in l1.  The last policy's reward vector is NaN:
    every q under it is NaN, so its a* is 0, and l1 and the psi update stay finite."""
    N, B = BATCHES[batch]
    gen = torch.Generator().manual_seed(21)
    sf = build(precision, N)
    lib = sf._library
    w = torch.zeros(D)
    w[:2] = 1.0
    e = torch.eye(D)
    wnan = w.clone()
    wnan[0] = NAN
    ws = [w] * (N - 1) + [wnan]
    nets = []
    for p in range(N):
        bo = torch.zeros(A, D)
        bo[0] = 2.0 * e[2]                           # action 0: q = 0, a psi row of its own
        bo[6 - p] = e[0]                             # policy p holds the maximum q = 1 at actions 6 - p and 8 - p:
        bo[8 - p] = e[1]                             # the key's a* is 6 - (N - 1), held by the last policy only
        Wo = torch.randint(-1, 2, (A * D, S), generator=gen).float() * (torch.rand(A * D, S, generator=gen) < 0.1)
        Wo[:, :] *= (torch.arange(A * D) % D >= 2).float()[:, None]      # the state moves psi only off the q-carrying features
        nets.append((Wo, bo.reshape(-1)))
        load_exact(sf, p, Wo, bo.reshape(-1), ws[p])
    tr = list(wl.synthetic_transitions(B, S, A, D, gen))
    tr[0], tr[4] = exact_states(B, gen), exact_states(B, gen)
    q_next = [q64(nets, tr[4], ws[i]) for i in range(N)]
    next_a = [gu.gpi_rule(q_next[i].reshape(B, -1), torch.arange(A).repeat(N))[0] for i in range(N)]
    assert int((next_a[0] == 6 - (N - 1)).sum()) == B and int((next_a[N - 1] == 0).sum()) == B
    steps = range(N) if policy == 'single' else [None]
    for i in steps:
        if i is None:
            losses = sf.update_successor_all(gu.cuda_tr(tr), True).cpu().double()
            idx = range(N)
        else:
            losses = torch.stack([torch.as_tensor(float(v)) for v in sf.update_successor(gu.cuda_tr(tr), i, True)]).double()[None]
            idx = [i]
        for row, j in enumerate(idx):
            l1, l2 = td_reference(nets, tr, j, ws[j], next_a[j])
            msg = f'{precision} {batch} {policy} policy {j}'
            assert abs(float(losses[row, 1]) - l1) <= 1e-5 * l1, (msg, 'l1', float(losses[row, 1]), l1)
            if j < N - 1:
                assert abs(float(losses[row, 2]) - l2) <= 1e-5 * l2, (msg, 'l2', float(losses[row, 2]), l2)
            for W, b in gu.psi_params(sf, j):
                assert bool(W.isfinite().all()) and bool(b.isfinite().all()), (msg, 'the psi update is not finite')
        if i is not None:                                # the next policy's step starts from the tables again
            for p, (Wo, bo) in enumerate(nets):
                load_exact(sf, p, Wo, bo, ws[p])
