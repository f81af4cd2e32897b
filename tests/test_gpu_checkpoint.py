"""
-m gpu: checkpoints of the packed SF libraries and the agents (state_dict / load_state_dict).  A run that is saved, restored
into a freshly built object (other weights, other seed) and continued must compute what the uninterrupted run computes, bit
for bit, in every precision mode: the master weights are fp32 everywhere and everything derived (operand shadows, step plans,
Adam bias corrections) is rebuilt on load from the saved state.
"""
import copy
import io
import random
import types

import numpy as np
import pytest
import torch

from oracle.sf_oracle import synthetic_transitions
from tests import gpu_util as gu
from tests.golden_util import load, rel_err
from tests.test_gpu_agent import build_agent
from tests.test_gpu_autograd import PRECISIONS, STEP_TOL, eager_g2_update, hyper, make_oracle
from deep_successor_features_for_transfer_b200 import ensemble, sfdqn, sfdqn_phi, tsfdqn_nf
from deep_successor_features_for_transfer_b200.workloads import ENVS, ShapeTask, build_sf_library, build_tsf_agent, model_lambda

pytestmark = pytest.mark.gpu
S, A, D = ENVS['reacher']['S'], ENVS['reacher']['A'], ENVS['reacher']['D']
N, B, EV = 3, 256, 5                       # target_update_ev 5: a target sync falls inside the resumed steps


def roundtrip(sd):
    buf = io.BytesIO()
    torch.save(sd, buf)
    buf.seek(0)
    return torch.load(buf)


def lib_tensors(lib):
    out = {k: getattr(lib, k).detach()[:lib.n] for k in lib._state_rows()}
    if lib.G is not None:
        out['h'] = lib.h
    return out


def assert_libs_equal(a, b):
    ta, tb = lib_tensors(a), lib_tensors(b)
    for k in ta:
        assert torch.equal(ta[k], tb[k]), f"'{k}' differs: max |diff| {float((ta[k].double() - tb[k].double()).abs().max())}"


def gpi_keys(sf, x):
    return [torch.cat(sf._library.gpi(x, sf._library.w[i])[1:]) for i in range(sf.n_tasks)]


# ---- builders: (SF object, step function) of each generation -------------------------------------------------------------------
def build(case, precision, seed):
    """case: 'g2' single-policy steps, 'g1' ensemble update_successors, 'g3' TSF with beta = 30, 'nf' TSF with 3 planar flows."""
    if case == 'g2':
        sf = build_sf_library('reacher', N, precision=precision, seed=seed, target_update_ev=EV)
        return sf, lambda tr, k: torch.stack(list(sf.update_successor(tr, k % N, True)))
    if case == 'g1':
        torch.manual_seed(seed)
        sf = ensemble.DeepSF(model_lambda([256, 256], ['relu', 'relu']), target_update_ev=EV,
                             hyperparameters=dict(gu.HYPER, precision=precision))
        sf.reset()
        for i in range(N):
            sf.add_training_task(ShapeTask(S, A, D, i))
        return sf, lambda tr, k: sf.update_successors(tr[:2] + tr[3:]).clone()
    if case == 'g3':
        sf, ag = build_tsf_agent('reacher', N, beta=30, precision=precision, seed=seed, target_update_ev=EV)
    else:
        torch.manual_seed(seed)
        hp = dict(gu.HYPER, g_h_function_dims=100, beta_loss_coefficient=1, n_coupling_layers=3, precision=precision)
        sf = tsfdqn_nf.DeepTSF(model_lambda([256, 256], ['relu', 'relu']), target_update_ev=EV, hyperparameters=hp)
        ag = tsfdqn_nf.TSFDQN(deep_sf=sf, buffer_handle=lambda: tsfdqn_nf.ReplayBuffer(), gamma=0.9, T=500, encoding=None,
                              hyperparameters=hp)
        ag.reset()
        for i in range(N):
            ag.add_training_task(ShapeTask(S, A, D, i))
    return sf, lambda tr, k: torch.stack(list(ag.update_successor(tr, k % N, True)))


def batches(n, seed):
    gen = torch.Generator().manual_seed(seed)
    return [gu.cuda_tr(synthetic_transitions(B, S, A, D, gen)) for _ in range(n)]


def resume_and_compare(case, precision, step_a, before_save=None, k1=7, k2=8):
    """A: k1 steps, save, k2 steps.  B (other seed): load, the same k2 steps; then every buffer, loss and GPI key is equal."""
    sf_a, step = build(case, precision, seed=1)
    tr1, tr2 = batches(k1, 100), batches(k2, 200)
    for k, tr in enumerate(tr1):
        step_a(sf_a, step, tr, k)
    assert any(u for u in sf_a.updates_since_target_updated)
    if before_save is not None:
        before_save(sf_a)
    sd = roundtrip(sf_a.state_dict())
    la = [step_a(sf_a, step, tr, k1 + k) for k, tr in enumerate(tr2)]
    sf_b, step2 = build(case, precision, seed=2)
    assert not torch.equal(sf_b._library.online[:N], sf_a._library.online[:N])
    sf_b.load_state_dict(sd)
    lb = [step_a(sf_b, step2, tr, k1 + k) for k, tr in enumerate(tr2)]
    for k, (x, y) in enumerate(zip(la, lb)):
        assert torch.equal(x, y), f'losses of resumed step {k} differ: {x.tolist()} vs {y.tolist()}'
    assert_libs_equal(sf_a._library, sf_b._library)
    assert sf_a.updates_since_target_updated == sf_b.updates_since_target_updated
    probe = batches(1, 300)[0][4]
    for ka, kb in zip(gpi_keys(sf_a, probe), gpi_keys(sf_b, probe)):
        assert torch.equal(ka, kb)


# ---- 1. bit-exact resume ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('case', ['g2', 'g1', 'g3', 'nf'])
def test_resume_is_bit_exact(case, precision):
    resume_and_compare(case, precision, lambda sf, step, tr, k: step(tr, k))


# ---- 2. out-of-phase Adam parity survives a checkpoint ---------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_resume_with_out_of_phase_bias_corrections(precision):
    def mixed(sf, step, tr, k):                     # single-policy and all-policy steps interleaved
        return sf.update_successor_all(tr).clone() if k % 3 == 1 else step(tr, k)

    def out_of_phase(sf):
        assert len(set(sf._library._adam_par[:N])) > 1

    resume_and_compare('g2', precision, mixed, before_save=out_of_phase)


# ---- 3. eager and fused steps mixed ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_resume_with_eager_and_fused_steps(precision):
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N, target_update_ev=EV)
    i = 1

    def build_ag(seed):
        o, _ = make_oracle(S, A, D, N, seed=seed)
        return gu.build_g2(meta, oracle=o, hyper=hyper(precision))

    def step(sf, tr, k):
        out = eager_g2_update(sf, tr, i, True) if k % 2 else sf.update_successor(tr, i, True)
        return torch.stack(list(out))

    sf_a = build_ag(1)
    tr1, tr2 = batches(3, 100), batches(6, 200)
    for k, tr in enumerate(tr1):
        step(sf_a, tr, k)
    sd = roundtrip(sf_a.state_dict())
    la = [step(sf_a, tr, 3 + k) for k, tr in enumerate(tr2)]
    sf_b = build_ag(2)
    psi = sf_b.get_successors(tr1[0][0])
    sf_b.load_state_dict(sd)
    with pytest.raises(RuntimeError, match='modified'):
        psi.sum().backward()
    lb = [step(sf_b, tr, 3 + k) for k, tr in enumerate(tr2)]
    for x, y in zip(la, lb):
        assert torch.equal(x, y)
    assert_libs_equal(sf_a._library, sf_b._library)


# ---- 4. the checkpoint does not depend on the precision mode ---------------------------------------------------------------------
def test_cross_precision_load_and_larger_capacity():
    sf_a, step = build('g2', 'bf16', seed=1)
    for k, tr in enumerate(batches(4, 100)):
        step(tr, k)
    x = batches(1, 300)[0][0]
    bf16_fwd = sf_a.get_successors(x)
    sd = roundtrip(sf_a.state_dict())
    ref = build_sf_library('reacher', N, precision='fp32', seed=3)          # fp32, the same weights through the module views
    for i in range(N):
        gu.load_policy(ref, i, gu.psi_params(sf_a, i), sf_a.fit_w[i].weight.data.cpu())
    fp32 = build_sf_library('reacher', N, precision='fp32', seed=2)
    fp32.load_state_dict(sd)
    assert torch.equal(fp32.get_successors(x), ref.get_successors(x))
    back = build_sf_library('reacher', N, precision='bf16', seed=4)
    back.get_successors(x)                                                  # shadows packed from the old weights
    back.load_state_dict(roundtrip(fp32.state_dict()))
    assert torch.equal(back.get_successors(x), bf16_fwd)
    big = build_sf_library('reacher', N, precision='fp32', seed=5)
    big._library._alloc(16)
    big.load_state_dict(sd)
    assert big._library.cap == 16
    assert torch.equal(big.get_successors(x), ref.get_successors(x))
    tr = batches(1, 400)[0]
    assert torch.equal(torch.stack(list(big.update_successor(tr, 0))), torch.stack(list(fp32.update_successor(tr, 0))))


# ---- 5. interop with the reference's eager objects -----------------------------------------------------------------------------
def reference_from_checkpoint(sd, i):
    """The reference's eager objects for every task (psi_model, target, fit_w) and a stock torch.optim.Adam for task i, loaded
    from an SF state_dict."""
    from deep_successor_features_for_transfer_b200.library import NetSpec
    handle = model_lambda([256, 256], ['relu', 'relu'])
    lsd = sd['library']
    ref = types.SimpleNamespace(psi=[], fit_w=[], updates_since_target_updated=list(sd['updates_since_target_updated']),
                                target_update_ev=sd['target_update_ev'])
    for j in range(sd['n_tasks']):
        model, _, _ = handle(S, A * D, (A, D), 1)
        target, _, _ = handle(S, A * D, (A, D), 1)
        model, target = model.cuda(), target.cuda()
        model.load_state_dict(sd['psi'][j]['model'])
        spec, _ = NetSpec.from_module(target, A, D)
        flat = [t for Wb in spec.views(lsd['target'][j]) for t in Wb]
        target.load_state_dict(dict(zip(target.state_dict().keys(), flat)))
        w = torch.nn.Linear(D, 1, bias=False, device='cuda')
        with torch.no_grad():
            w.weight.copy_(lsd['w'][j].view(1, -1))
        optim = None
        if j == i:
            optim = torch.optim.Adam([{'params': model.parameters(), 'lr': 1e-3, 'weight_decay': 0},
                                      {'params': w.parameters(), 'lr': 1e-3, 'weight_decay': 0}])
            optim.load_state_dict(sd['psi'][j]['optim'])
        ref.psi.append(((model, None, optim), (target, None, None)))
        ref.fit_w.append(w)

    def GPI(x, task):
        with torch.no_grad():
            psis = torch.stack([m(x) for (m, _, _), _ in ref.psi], dim=1)          # [B, N, A, D]
            return psis @ ref.fit_w[task].weight.view(-1), None
    ref.GPI = GPI
    return ref


def test_reference_interop_both_directions():
    i, K = 1, 10
    sf, _ = build('g2', 'fp32', seed=1)
    for k, tr in enumerate(batches(3, 100)):
        sf.update_successor(tr, k % N)
    sd = roundtrip(sf.state_dict())
    ref = reference_from_checkpoint(sd, i)
    (model, _, optim), _ = ref.psi[i]
    assert int(optim.state_dict()['state'][0]['step']) == int(sf._library.step[i])
    for k, tr in enumerate(batches(K, 200)):
        got = sf.update_successor(tr, i, True)
        want = eager_g2_update(ref, tr, i, True)
        assert np.allclose([float(v) for v in got], [float(v) for v in want], rtol=2e-5, atol=1e-8), k
    st = sf.psi[i][0][2].state
    ost = optim.state
    for lin, rlin in zip(gu.linears(sf.psi[i][0][0].net), gu.linears(model)):
        for p, rp in ((lin.weight, rlin.weight), (lin.bias, rlin.bias)):
            assert rel_err(p.data.cpu(), rp.data.cpu()) < STEP_TOL
            assert rel_err(st[p]['exp_avg'].cpu(), ost[rp]['exp_avg'].cpu()) < 2e-5
            assert rel_err(st[p]['exp_avg_sq'].cpu(), ost[rp]['exp_avg_sq'].cpu()) < 4e-5
    assert rel_err(sf.fit_w[i].weight.data.cpu(), ref.fit_w[i].weight.data.cpu()) < STEP_TOL
    assert sf.updates_since_target_updated[i] == ref.updates_since_target_updated[i]

    # the other way: the stock optimizer's state (and the eager weights) into the packed library
    packed = sf.psi[i][0][2]
    with torch.no_grad():
        for lin, rlin in zip(gu.linears(sf.psi[i][0][0].net), gu.linears(model)):
            lin.weight.copy_(rlin.weight)
            lin.bias.copy_(rlin.bias)
        sf.fit_w[i].weight.copy_(ref.fit_w[i].weight)
    packed.load_state_dict(optim.state_dict())
    st = packed.state
    assert int(sf._library.step[i]) == int(ost[model[0].weight]['step'])
    for lin, rlin in zip(gu.linears(sf.psi[i][0][0].net), gu.linears(model)):
        for p, rp in ((lin.weight, rlin.weight), (lin.bias, rlin.bias)):
            assert torch.equal(st[p]['exp_avg'], ost[rp]['exp_avg']) and torch.equal(st[p]['exp_avg_sq'], ost[rp]['exp_avg_sq'])
    assert torch.equal(st[sf.fit_w[i].weight]['exp_avg'], ost[ref.fit_w[i].weight]['exp_avg'])
    tr = batches(1, 500)[0]
    got, want = sf.update_successor(tr, i, True), eager_g2_update(ref, tr, i, True)
    assert np.allclose([float(v) for v in got], [float(v) for v in want], rtol=2e-5, atol=1e-8)
    for lin, rlin in zip(gu.linears(sf.psi[i][0][0].net), gu.linears(model)):
        assert rel_err(lin.weight.data.cpu(), rlin.weight.data.cpu()) < STEP_TOL


# ---- 6. replay rings and agents ------------------------------------------------------------------------------------------------
def test_replay_rings_exchange_state():
    task = toy_task(11)
    host = sfdqn.ReplayBuffer(n_samples=50, n_batch=16)
    s = task.initialize()
    for _ in range(70):                                           # wrapped: the write index is not the size
        a = random.randrange(task.A)
        s1, r, done = task.transition(a)
        host.append(s, torch.tensor(a), r, task.features(s, a, s1), s1, 0.0 if done else 0.9)
        s = task.initialize() if done else s1
    dev = sfdqn.DeviceReplayBuffer(n_samples=50, n_batch=16)
    dev.load_state_dict(roundtrip(host.state_dict()))
    host2 = sfdqn.ReplayBuffer(n_samples=50, n_batch=16)
    host2.load_state_dict(roundtrip(dev.state_dict()))
    assert (dev.index, dev.size, host2.index, host2.size) == (20, 50, 20, 50)
    outs = []
    for ring in (host, dev, host2):
        np.random.seed(5)
        outs.append([t.clone() for t in ring.replay()])
    for other in outs[1:]:
        for x, y in zip(outs[0], other):
            assert torch.equal(x.reshape(y.shape).to(y.dtype), y)


def toy_task(seed):
    from tests.toy_task import ToyTask
    return ToyTask(4, 5, 6, 0, seed=seed)


@pytest.mark.parametrize('name,device_ring', [('agent_sfdqn_toy', False), ('agent_tsfdqn_toy', True)])
def test_agent_resume(name, device_ring):
    meta, z = load(name)
    k1, k2 = 60, 40

    def run(ag, tasks, holder, n, task_index, first):
        losses, inner = [], holder.update_successor

        def recording(transitions, policy_index, use_gpi=True):
            res = inner(transitions, policy_index, use_gpi)
            losses.append(None if res is None else torch.stack(list(res)))
            return res
        holder.update_successor = recording
        if first:
            ag.set_active_training_task(task_index)
        for _ in range(n):
            ag.next_sample(None, None)
            ag.total_training_steps += 1
        holder.update_successor = inner
        return losses

    def holder_of(sf, ag):
        return ag if meta['kind'] == 'agent_tsfdqn' else sf

    sf_a, ag_a, tasks_a = build_agent(meta, z, device_ring)
    random.seed(meta['seed'])
    np.random.seed(meta['seed'])
    torch.manual_seed(meta['seed'])
    run(ag_a, tasks_a, holder_of(sf_a, ag_a), k1, 0, True)
    sd = roundtrip(ag_a.state_dict())
    rng = (random.getstate(), np.random.get_state(), torch.get_rng_state())     # the caller's, as in torch
    envs = copy.deepcopy(tasks_a)                                                 # and so are the environments
    la = run(ag_a, tasks_a, holder_of(sf_a, ag_a), 100 - k1, 0, False) + run(ag_a, tasks_a, holder_of(sf_a, ag_a), k2, 1, True)

    sf_b, ag_b, _ = build_agent(meta, z, device_ring)
    with torch.no_grad():
        sf_b._library.online.add_(0.01)
        sf_b._library.w.add_(0.01)
    ag_b.tasks, ag_b.phis = envs, [t.features for t in envs]
    ag_b.load_state_dict(sd)
    random.setstate(rng[0])
    np.random.set_state(rng[1])
    torch.set_rng_state(rng[2])
    lb = run(ag_b, envs, holder_of(sf_b, ag_b), 100 - k1, 0, False) + run(ag_b, envs, holder_of(sf_b, ag_b), k2, 1, True)

    for ta, tb in zip(tasks_a, envs):
        assert ta.actions_taken == tb.actions_taken
    assert len(la) == len(lb) and all((x is None and y is None) or torch.equal(x, y) for x, y in zip(la, lb))
    assert sum(x is not None for x in la) > 50
    for ca, cb in zip(sf_a.gpi_counters, sf_b.gpi_counters):
        assert np.array_equal(ca, cb)
    assert_libs_equal(sf_a._library, sf_b._library)
    assert sf_a.updates_since_target_updated == sf_b.updates_since_target_updated
    assert ag_a.total_training_steps == ag_b.total_training_steps and ag_a.epsilon == ag_b.epsilon
    assert float(ag_a.cum_reward) == float(ag_b.cum_reward)


def test_target_task_state_roundtrip():
    """TSFDQN's target tasks: the fused optimizer's moments / counters and omega come back; the eager kind too."""
    target_hp = dict(learning_rate_omega=1e-2, weight_decay_omega=0.0, learning_rate_omega_decay=0.05, omegas_l1_coefficient=0.1)
    sf, ag = build_tsf_agent('reacher', 2, seed=1)
    ag.hyperparameters.update(target_hp)
    omegas0 = torch.full((1, 2, 1, 1), 0.5, device='cuda')
    for fused in (True, False):
        ag.test_tasks_weights, ag.omegas = [], []
        w, optim, sched, om = ag._new_target_task(D, omegas0, fused=fused)
        ag.test_tasks_weights.append((w, optim, sched))
        ag.omegas.append(om)
        task = ShapeTask(S, A, D, 0)
        task.features = lambda s, a, s1: torch.linspace(0, 1, D)
        for _ in range(3):
            s, s1 = torch.randn(1, S, device='cuda'), torch.randn(1, S, device='cuda')
            ag.update_test_reward_mapper(w, om, optim, task, 0.5, s, 1, s1, 2)
            sched.step()
        sd = roundtrip(ag.state_dict())
        _, ag2 = build_tsf_agent('reacher', 2, seed=2)
        ag2.hyperparameters.update(target_hp)
        ag2.load_state_dict(sd)
        w2, optim2, sched2 = ag2.test_tasks_weights[0]
        assert torch.equal(w2.weight, w.weight) and torch.equal(ag2.omegas[0], om)
        if fused:
            for k in ('w_m', 'w_v', 'o_m', 'o_v', 'counters'):
                assert torch.equal(getattr(optim2, k), getattr(optim, k))
        else:
            assert sched2.last_epoch == sched.last_epoch == 3
            assert optim2.param_groups[1]['lr'] == optim.param_groups[1]['lr']
            for p, p2 in zip([w.weight, om], [w2.weight, ag2.omegas[0]]):
                assert torch.equal(optim.state[p]['exp_avg'], optim2.state[p2]['exp_avg'])


# ---- 7. errors -------------------------------------------------------------------------------------------------------------------
def test_checkpoint_errors():
    sf, step = build('g2', 'fp32', seed=1)
    for k, tr in enumerate(batches(2, 100)):
        step(tr, k)
    sd = roundtrip(sf.state_dict())
    narrow = build_sf_library('reacher', N, hidden=(128, 128), seed=2)
    with pytest.raises(ValueError, match="'dims'"):
        narrow.load_state_dict(sd)
    fewer = build_sf_library('reacher', N - 1, seed=2)
    with pytest.raises(ValueError, match='tasks'):
        fewer.load_state_dict(sd)
    with pytest.raises(ValueError, match='policies'):
        fewer._library.load_state_dict(sd['library'])
    newer = copy.copy(sd['library'])
    newer['version'] = 99
    with pytest.raises(ValueError, match='newer'):
        sf._library.load_state_dict(newer)
    missing = {k: v for k, v in sd['library'].items() if k != 'm'}
    with pytest.raises(ValueError, match="missing key 'm'"):
        sf._library.load_state_dict(missing)
    osd = copy.deepcopy(sd['psi'][0]['optim'])
    osd['state'][0]['step'] = torch.tensor(99.0)
    with pytest.raises(ValueError, match='different Adam steps'):
        sf.psi[0][0][2].load_state_dict(osd)
    osd = copy.deepcopy(sd['psi'][0]['optim'])
    del osd['state'][1]
    with pytest.raises(ValueError, match='only some parameters'):
        sf.psi[0][0][2].load_state_dict(osd)
    lib = sf._library
    lib.shard = types.SimpleNamespace(world=2)
    with pytest.raises(NotImplementedError):
        lib.state_dict()
    with pytest.raises(NotImplementedError):
        lib.load_state_dict(sd['library'])
    lib.shard = None
    phi = sfdqn_phi.DeepSF_PHI(model_lambda([256, 256], ['relu', 'relu']), hyperparameters=dict(gu.HYPER))
    with pytest.raises(NotImplementedError):
        phi.state_dict()
    with pytest.raises(NotImplementedError):
        phi.load_state_dict(sd)
    sf.load_state_dict(sd)                                     # a failed load changed nothing it could not restore
    assert_libs_equal(sf._library, build_and_load(sd))


def build_and_load(sd):
    sf = build_sf_library('reacher', N, seed=3)
    sf.load_state_dict(sd)
    return sf._library
