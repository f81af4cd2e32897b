"""
-m gpu: autograd through the packed psi networks (PackedSFLibrary.psi, DeepSF(autograd=True)) and the eager optimizer step
(PackedAdamView.step / zero_grad).  The backward kernels run with a DENSE dL/dpsi [B][n_pol][A*D] (actions == NULL in the C ABI).
Bounds are the ones of the existing backward / golden tests this file mirrors:
  dense gradients vs torch autograd      test_psi_backward_vs_autograd (tests/test_gpu_bf16.py, tests/test_gpu_tf32.py)
  eager reference update vs the goldens  test_g2_update_successor_vs_golden / test_g3_tsf_vs_golden (tests/test_gpu_parity.py),
                                         test_tf32x3_update_successor_vs_golden_h256 (tests/test_gpu_tf32.py)
"""
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle.sf_oracle import OracleSF, act_fn, synthetic_transitions
from tests import gpu_util as gu
from tests.golden_util import load, n_layers, rel_err, t, transitions
from tests.test_gpu_bf16 import _rb
from tests.test_gpu_tf32 import MOMENT_TOL, relu_kink_rows, weights_close

pytestmark = pytest.mark.gpu
FWD_TOL, STEP_TOL = 1e-5, 1e-4
PRECISIONS = ['fp32', 'bf16', 'tf32', 'tf32x3']


def fro_err(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def mean_err(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).abs().mean() / b.abs().max().clamp_min(1e-30))


def make_oracle(S, A, D, N, seed, tsf_dim=None):
    gen = torch.Generator().manual_seed(seed)
    o = OracleSF(S, A, D, (256, 256), ('relu', 'relu'), tsf_dim=tsf_dim)
    for _ in range(N):
        o.add_random_policy(gen)
    return o, gen


def hyper(precision='fp32', autograd=True, **kw):
    return dict(gu.HYPER, precision=precision, autograd=autograd, **kw)


def build_g3(meta, z=None, oracle=None):
    """tests/gpu_util.build_g3 with autograd=True."""
    from deep_successor_features_for_transfer_b200.tsfdqn import DeepTSF, TSFDQN, ReplayBuffer
    hp = hyper(g_h_function_dims=meta['gdim'], beta_loss_coefficient=meta['beta'])
    dsf = DeepTSF(pytorch_model_handle=gu.model_lambda(meta['hidden'], meta['acts']), use_true_reward=False,
                  target_update_ev=meta.get('target_update_ev', 1000), hyperparameters=hp)
    ag = TSFDQN(deep_sf=dsf, buffer_handle=lambda: ReplayBuffer(), gamma=0.9, T=500, encoding=None,
                use_gpi=meta.get('use_gpi', True), hyperparameters=hp)
    ag.reset()
    for i in range(meta['N']):
        ag.add_training_task(gu.FakeTask(meta['S'], meta['A'], meta['D'], i))
    with torch.no_grad():
        for i in range(meta['N']):
            if z is not None:
                layers = [(t(z[f'init.psi{i}.W{l}']), t(z[f'init.psi{i}.b{l}'])) for l in range(n_layers(meta))]
                gu.load_policy(dsf, i, layers, t(z[f'init.w{i}']))
                gW, gb = t(z[f'init.g{i}.W']), t(z[f'init.g{i}.b'])
            else:
                gu.load_policy(dsf, i, oracle.psi[i], oracle.w[i])
                gW, gb = oracle.g[i]
            ag.g_functions[i].weight.data.copy_(gW)
            ag.g_functions[i].bias.data.copy_(gb)
        hW, hb = (t(z['init.h.W']), t(z['init.h.b'])) if z is not None else oracle.h
        ag.h_function.weight.data.copy_(hW)
        ag.h_function.bias.data.copy_(hb)
    return dsf, ag


# ---- the reference's update bodies, restated in plain torch on the packed library ---------------------------------------------
def _next_actions(sf, psi_model, next_states, i, use_gpi):
    if use_gpi:
        q1, _ = sf.GPI(next_states, i)
        return torch.argmax(torch.max(q1, dim=1).values, dim=-1)
    q1 = sf.fit_w[i](psi_model(next_states))
    return torch.squeeze(torch.argmax(q1, dim=1), dim=1)


def _target_sync(sf, i, psi_model, target_psi_model):
    sf.updates_since_target_updated[i] += 1
    if sf.updates_since_target_updated[i] >= sf.target_update_ev:
        target_psi_model.load_state_dict(psi_model.state_dict())
        sf.updates_since_target_updated[i] = 0


def eager_g2_update(sf, transitions, i, use_gpi=True):
    """sfdqn.py:303-371."""
    states, actions, rs, phis, next_states, gammas = transitions
    (psi_model, _, optim), (target_psi_model, _, _) = sf.psi[i]
    B = len(gammas)
    idx = torch.arange(B, device=states.device)
    gammas = gammas.reshape(-1, 1)
    with torch.no_grad():
        next_actions = _next_actions(sf, psi_model, next_states, i, use_gpi)
        targets = phis + gammas * target_psi_model(next_states)[idx, next_actions, :]
    current_psi = psi_model(states)
    merge = current_psi.clone()
    merge[idx, actions, :] = targets
    l1 = F.mse_loss(current_psi, merge)
    l2 = F.mse_loss(sf.fit_w[i](phis), rs)
    loss = l1 + l2
    optim.zero_grad()
    loss.backward()
    optim.step()
    _target_sync(sf, i, psi_model, target_psi_model)
    return loss.detach(), l1.detach(), l2.detach()


def eager_g3_update(ag, transitions, i, use_gpi=True):
    """tsfdqn.py:588-709."""
    sf = ag.sf
    states, actions, rs, phis, next_states, gammas = transitions
    (psi_model, _, optim), (target_psi_model, _, _) = sf.psi[i]
    g_function, h_function = ag.g_functions[i], ag.h_function
    B = len(gammas)
    idx = torch.arange(B, device=states.device)
    gammas = gammas.reshape(-1, 1)
    with torch.no_grad():
        next_actions = _next_actions(sf, psi_model, next_states, i, use_gpi)
        next_psis = target_psi_model(next_states)[idx, next_actions, :]
    current_psi = psi_model(states)
    aff = h_function(g_function(states)) + h_function(g_function(next_states))
    tphis = aff * phis
    targets = tphis + gammas * next_psis
    merge = current_psi.clone()
    merge[idx, actions, :] = targets
    l1 = F.mse_loss(current_psi, merge)
    l2 = F.mse_loss(sf.fit_w[i](tphis), rs)
    loss = l1 + torch.tensor(ag.hyperparameters['beta_loss_coefficient'], device=states.device) * l2
    optim.zero_grad()
    loss.backward()
    optim.step()
    _target_sync(sf, i, psi_model, target_psi_model)
    return loss.detach(), l1.detach(), l2.detach()


# ---- 1. forward unchanged -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_recorded_forward_equals_plain_forward(precision):
    S, A, D, N, B = 4, 9, 12, 3, 1000
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make_oracle(S, A, D, N, seed=3)
    sf = gu.build_g2(meta, oracle=o, hyper=hyper(precision))
    plain = gu.build_g2(meta, oracle=o, hyper=hyper(precision, autograd=False))
    x = synthetic_transitions(B, S, A, D, gen)[0].cuda()
    psi = sf.get_successors(x)
    assert psi.requires_grad
    with torch.no_grad():
        ref = sf.get_successors(x)
    assert not ref.requires_grad
    assert torch.equal(psi.detach(), ref)
    assert torch.equal(ref, plain.get_successors(x))
    assert torch.equal(sf.get_successor(x, 1).detach(), plain.get_successor(x, 1))
    assert torch.equal(sf.psi[2][0][0](x).detach(), plain.psi[2][0][0](x))


# ---- 2. dense gradients against torch autograd ----------------------------------------------------------------------------------
def torch_dense_grads(o, pol, x, G, emulate_bf16=False):
    rb = _rb if emulate_bf16 else (lambda v: v)
    layers = [(W.clone().requires_grad_(True), b.clone().requires_grad_(True)) for W, b in o.psi[pol]]
    h = rb(x)
    for (W, b), a in zip(layers, o.acts):
        h = act_fn(a)(torch.addmm(b, h, rb(W).t()))
        if W is not layers[-1][0]:
            h = rb(h)
    (h.view(x.shape[0], o.A, o.D) * G).sum().backward()
    return [(W.grad, b.grad) for W, b in layers]


# tf32x3: 2e-5, not the sparse test's 1e-5.  With a dense dL/dpsi every output column feeds the reductions, and the error of the
# tensor cores' fp32 accumulation grows with their length: measured 4e-6 .. 5e-6 at B = 1000, 0.9e-5 .. 1.1e-5 at B = 4219 and
# 1.2e-5 .. 1.3e-5 at Hopper's 1350 columns, the same with a float64 autograd reference and with a 10x wider ReLU-kink band.
# The dense kernels' own contribution is nil: test_dense_gradient_equals_sparse shows them bit-identical to the sparse ones.
@pytest.mark.parametrize('precision,tol', [('fp32', 2e-5), ('bf16', 1.5e-2), ('tf32x3', 2e-5), ('tf32', 6e-2)])
@pytest.mark.parametrize('S,A,D,N,B,hopper', [
    (4, 9, 12, 3, 1000, False),
    (4, 9, 12, 5, 33 * 128 - 5, False),
    (11, 27, 50, 2, 300, True),
    (4, 2, 20, 2, 32, False),
])
def test_dense_backward_vs_autograd(precision, tol, S, A, D, N, B, hopper):
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make_oracle(S, A, D, N, seed=77)
    sf = gu.build_g2(meta, oracle=o, hyper=hyper(precision))
    x = synthetic_transitions(B, S, A, D, gen, hopper=hopper)[0]
    G = torch.randn(B, N - 1, A, D, generator=gen) * 1e-4
    if precision == 'tf32x3':
        for p in range(N - 1):
            G[relu_kink_rows(o, 1 + p, x), p] = 0.0
    (sf.get_successors(x.cuda())[:, 1:] * G.cuda()).sum().backward()
    for lin in gu.linears(sf.psi[0][0][0].net):                    # policy 0 is outside the loss
        assert lin.weight.grad is None or not lin.weight.grad.any()
    for p in range(1, N):
        ref = torch_dense_grads(o, p, x, G[:, p - 1], emulate_bf16=precision == 'bf16')
        for l, (lin, (gW, gb)) in enumerate(zip(gu.linears(sf.psi[p][0][0].net), ref)):
            assert fro_err(lin.weight.grad, gW) < tol, f'policy {p} layer {l}: dW error {fro_err(lin.weight.grad, gW)}'
            assert fro_err(lin.bias.grad, gb) < tol, f'policy {p} layer {l}: db error {fro_err(lin.bias.grad, gb)}'


# ---- 3. dense equals sparse -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('S,A,D,N,B,hopper', [(4, 9, 12, 3, 1000, False), (11, 27, 50, 2, 300, True)])
def test_dense_gradient_equals_sparse(precision, S, A, D, N, B, hopper):
    """A dense dL/dpsi that is zero outside psi[b, a_b, :] gives the train step's sparse gradient: the kernels build the same
    operand tiles.  fp32: the same FMA sequence over the same values (the zeros included), so equal as well."""
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make_oracle(S, A, D, N, seed=11)
    sf = gu.build_g2(meta, oracle=o, hyper=hyper(precision))
    lib = sf._library
    x, actions = (v.cuda() for v in synthetic_transitions(B, S, A, D, gen, hopper=hopper)[:2])
    lo, n_pol = 1, N - 1
    d_sel = (torch.randn(n_pol, B, D, generator=gen) * 1e-4).cuda()
    G = torch.zeros(B, n_pol, A, D, device='cuda')
    G[torch.arange(B, device='cuda'), :, actions, :] = d_sel.transpose(0, 1)
    (lib.psi(x, lo, n_pol) * G).sum().backward()
    dense = lib.online.grad[lo:lo + n_pol].clone()
    sparse = lib.psi_gradients(x, actions, d_sel, lo, n_pol)
    assert torch.equal(dense, sparse), float((dense - sparse).abs().max())


# ---- 4. the reference's update, restated in eager torch, meets the goldens ------------------------------------------------------
@pytest.mark.parametrize('name,precision', [('g2_reacher_gpi', 'fp32'), ('g2_reacher_sync', 'fp32'), ('g2_cartpole_tanh', 'fp32'),
                                            ('g2_hopper_gpi', 'fp32'), ('g2_reacher_h256', 'fp32'), ('g2_reacher_h256', 'tf32x3')])
def test_eager_g2_update_vs_golden(name, precision):
    meta, z = load(name)
    sf = gu.build_g2(meta, z, hyper=hyper(precision))
    i = meta['policy']
    for k in range(meta['K']):
        out = eager_g2_update(sf, gu.cuda_tr(transitions(z, k)), i, meta['use_gpi'])
        assert np.allclose([float(v) for v in out], z['out.losses'][k], rtol=2e-5, atol=1e-8)
    post, tgt = gu.psi_params(sf, i), gu.psi_params(sf, i, target=True)
    st = sf.psi[i][0][2].state
    lins = gu.linears(sf.psi[i][0][0].net)
    for l in range(n_layers(meta)):
        m, v = st[lins[l].weight]['exp_avg'].cpu(), st[lins[l].weight]['exp_avg_sq'].cpu()
        if precision == 'tf32x3':
            assert weights_close(post[l][0], z[f'post.psi.W{l}']) and weights_close(post[l][1], z[f'post.psi.b{l}'])
            assert rel_err(m, z[f'post.adam.W{l}.m']) < MOMENT_TOL and rel_err(v, z[f'post.adam.W{l}.v']) < MOMENT_TOL
            continue
        assert rel_err(post[l][0], z[f'post.psi.W{l}']) < STEP_TOL and mean_err(post[l][0], z[f'post.psi.W{l}']) < 2e-6
        assert rel_err(post[l][1], z[f'post.psi.b{l}']) < STEP_TOL
        assert rel_err(tgt[l][0], z[f'post.tgt.W{l}']) < STEP_TOL
        assert rel_err(m, z[f'post.adam.W{l}.m']) < 2e-5
        assert rel_err(v, z[f'post.adam.W{l}.v']) < 4e-5
        assert rel_err(st[lins[l].bias]['exp_avg'].cpu(), z[f'post.adam.b{l}.m']) < 2e-5
    assert rel_err(sf.fit_w[i].weight.data.cpu(), z['post.w']) < STEP_TOL
    assert int(sf._library.step[i]) == int(z['post.adam.w.step'])
    assert sf.updates_since_target_updated == list(z['post.updates_since_target_updated'])
    for j in range(meta['N']):
        if j != i:
            for l, (W, b) in enumerate(gu.psi_params(sf, j)):
                assert torch.equal(W, t(z[f'init.psi{j}.W{l}']))


@pytest.mark.parametrize('name', ['g3_reacher_gpi', 'g3_reacher_beta30'])
def test_eager_g3_update_vs_golden(name):
    meta, z = load(name)
    dsf, ag = build_g3(meta, z)
    for k in range(meta['K']):
        out = eager_g3_update(ag, gu.cuda_tr(transitions(z, k)), meta['policies'][k], meta['use_gpi'])
        assert np.allclose([float(v) for v in out], z['out.losses'][k], rtol=2e-5, atol=1e-8)
    stepped = sorted(set(meta['policies']))
    for i in stepped:
        for l, (W, b) in enumerate(gu.psi_params(dsf, i)):
            assert rel_err(W, z[f'post.psi{i}.W{l}']) < STEP_TOL
            assert rel_err(b, z[f'post.psi{i}.b{l}']) < STEP_TOL
        assert rel_err(dsf.fit_w[i].weight.data.cpu(), z[f'post.w{i}']) < STEP_TOL
        assert rel_err(ag.g_functions[i].weight.data.cpu(), z[f'post.g{i}.W']) < STEP_TOL
        assert rel_err(ag.g_functions[i].bias.data.cpu(), z[f'post.g{i}.b']) < STEP_TOL
        st = dsf.psi[i][0][2].state
        assert rel_err(st[ag.h_function.weight]['exp_avg'].cpu(), z[f'post.adam{i}.hW.m']) < 2e-5
        assert rel_err(st[ag.g_functions[i].weight]['exp_avg_sq'].cpu(), z[f'post.adam{i}.gW.v']) < 4e-5
        assert int(dsf._library.step[i]) == meta['policies'].count(i)
    assert rel_err(ag.h_function.weight.data.cpu(), z['post.h.W']) < STEP_TOL
    assert rel_err(ag.h_function.bias.data.cpu(), z['post.h.b']) < STEP_TOL
    for j in range(meta['N']):
        if j not in stepped:
            for l, (W, b) in enumerate(gu.psi_params(dsf, j)):
                assert torch.equal(W, t(z[f'init.psi{j}.W{l}']))


# ---- 5. eager and fused steps mixed ---------------------------------------------------------------------------------------------
def test_eager_and_fused_steps_mix():
    S, A, D, N, B, i = 4, 9, 12, 4, 4096, 2
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make_oracle(S, A, D, N, seed=5)
    sf = gu.build_g2(meta, oracle=o, hyper=hyper('fp32'))
    for k in range(4):
        tr = synthetic_transitions(B, S, A, D, gen)
        ref = o.update_successor(tr, i, True)
        trc = gu.cuda_tr(tr)
        out = eager_g2_update(sf, trc, i, True) if k % 2 == 0 else sf.update_successor(trc, i, True)
        assert np.allclose([float(v) for v in out], [float(v) for v in ref], rtol=2e-5, atol=1e-8)
    assert int(sf._library.step[i]) == 4
    st = sf.psi[i][0][2].state
    for l, (lin, (W, b)) in enumerate(zip(gu.linears(sf.psi[i][0][0].net), o.psi[i])):
        assert rel_err(lin.weight.data.cpu(), W) < STEP_TOL and rel_err(lin.bias.data.cpu(), b) < STEP_TOL
        assert rel_err(st[lin.weight]['exp_avg'].cpu(), o.adam[i]['m']['sf'][2 * l]) < STEP_TOL
        assert rel_err(st[lin.weight]['exp_avg_sq'].cpu(), o.adam[i]['v']['sf'][2 * l]) < STEP_TOL
    assert rel_err(sf.fit_w[i].weight.data.cpu(), o.w[i]) < STEP_TOL


# ---- 6. stock torch code sees the packed gradient ------------------------------------------------------------------------------
def test_stock_torch_optimizer_and_clipping_use_the_packed_gradient():
    S, A, D, N, B = 4, 9, 12, 3, 512
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make_oracle(S, A, D, N, seed=21)
    sf = gu.build_g2(meta, oracle=o, hyper=hyper('fp32'))
    lib = sf._library
    x = synthetic_transitions(B, S, A, D, gen)[0].cuda()
    G = torch.randn(B, A, D, device='cuda')
    model, _, optim = sf.psi[1][0]
    (model(x) * G).sum().backward()
    row0, grad0 = lib.online.detach()[1].clone(), lib.online.grad[1].clone()
    lr = 1e-3
    sgd = torch.optim.SGD(model.parameters(), lr=lr)
    sgd.zero_grad()                                                # set_to_none: the next backward starts afresh
    assert all(p.grad is None for p in model.parameters())
    (model(x) * G).sum().backward()
    assert torch.equal(lib.online.grad[1], grad0)
    assert all(p.grad is not None and p.grad.data_ptr() >= lib.online.grad.data_ptr() for p in model.parameters())
    sgd.step()
    assert torch.allclose(lib.online.detach()[1], row0 - lr * grad0, rtol=1e-6, atol=1e-9)
    optim.zero_grad()
    assert lib.online.grad[1].abs().sum() == 0 and all(p.grad is None for p in model.parameters())
    (model(x) * G).sum().backward()
    total = torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=1e-3)
    assert float(total) > 1e-3
    assert abs(float(lib.online.grad[1].norm()) - 1e-3) < 1e-8          # the packed row optim.step() reads was scaled
    w0 = lib.online.detach()[1].clone()
    optim.step()
    assert int(lib.step[1]) == 1 and not torch.equal(lib.online.detach()[1], w0)


# ---- 7. errors ------------------------------------------------------------------------------------------------------------------
def test_autograd_errors():
    S, A, D, N, B = 4, 9, 12, 3, 256
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make_oracle(S, A, D, N, seed=8)
    sf = gu.build_g2(meta, oracle=o, hyper=hyper('fp32'))
    lib = sf._library
    tr = gu.cuda_tr(synthetic_transitions(B, S, A, D, gen))
    x = tr[0]
    model, _, optim = sf.psi[1][0]
    psi = model(x)
    sf.update_successor(tr, 1, True)                               # the fused step moves the online rows
    with pytest.raises(RuntimeError):
        psi.sum().backward()
    with pytest.raises(ValueError):
        sf.get_successors(x.clone().requires_grad_())
    psi = model(x)
    d_psi = torch.ones_like(psi, requires_grad=True)
    with pytest.raises(RuntimeError):                              # no double backward
        torch.autograd.grad(psi, lib.online, d_psi, create_graph=True)[0].sum().backward()
    # an optimizer group with only some gradients
    optim.zero_grad()
    (model(x)).sum().backward()
    gu.linears(model.net)[0].bias.grad = None
    with pytest.raises(RuntimeError):
        optim.step()
    # a group skipped by an earlier step that now has gradients
    optim.zero_grad()
    model(x).sum().backward()
    optim.step()                                                   # w has no gradient: skipped
    optim.zero_grad()
    (model(x).sum() + sf.fit_w[1](tr[3]).sum()).backward()
    with pytest.raises(RuntimeError):
        optim.step()
    # a precision mode change between the forward and its backward (the saved activations have the forward's layout)
    for mode in ('bf16', 'tf32x3'):
        psi = lib.psi(x, 0, 2)
        lib.set_precision(mode)
        with pytest.raises(RuntimeError, match='precision'):
            psi.sum().backward()
        lib.set_precision('fp32')
    psi = lib.psi(x, 0, 2)
    lib.set_precision('bf16')
    lib.set_precision('fp32')
    psi.sum().backward()                                           # the same mode again: the saved layout is valid
    # a second backward without retain_graph: the saved activations were freed
    with pytest.raises(RuntimeError):
        psi.sum().backward()
    # sharded libraries
    lib.shard = types.SimpleNamespace(world=2)
    with pytest.raises(NotImplementedError):
        lib.psi(x, 0, 1)
    lib.shard = None
    # autograd=False: step() raises as before, and the forwards record nothing
    plain = gu.build_g2(meta, oracle=o, hyper=hyper('fp32', autograd=False))
    assert not plain.get_successors(x).requires_grad
    with pytest.raises(RuntimeError):
        plain.psi[0][0][2].step()


def test_target_forwards_do_not_record():
    meta, z = load('g3_reacher_gpi')
    dsf, ag = build_g3(meta, z)
    x = t(z['tr0.states']).cuda()
    assert dsf.get_successors(x).requires_grad
    assert not dsf.get_next_successors(x).requires_grad
    assert not dsf.get_next_successor(x, 0).requires_grad
    assert not dsf.psi[0][1][0](x).requires_grad
