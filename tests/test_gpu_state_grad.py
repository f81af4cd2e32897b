"""
-m gpu: gradients of the packed psi networks with respect to their input states (PackedSFLibrary(state_grad=True),
DeepSF(autograd=True, state_grad=True)): the backward returns dL/dx = sum_j dZ0_j . W0_j through sfgpi_mlp_input_grad.
Bounds are those of the dense weight-gradient test (tests/test_gpu_autograd.py::test_dense_backward_vs_autograd).
"""
import copy
import types

import numpy as np
import pytest
import torch

from oracle.sf_oracle import OracleSF, act_fn, synthetic_transitions
from tests import gpu_util as gu
from tests.golden_util import rel_err
from tests.test_gpu_autograd import PRECISIONS, STEP_TOL, eager_g2_update, eager_g3_update, fro_err, hyper
from tests.test_gpu_bf16 import _rb
from tests.test_gpu_tf32 import relu_kink_rows

pytestmark = pytest.mark.gpu


def make_oracle(S, A, D, N, seed, hidden=(256, 256), acts=('relu', 'relu'), tsf_dim=None):
    gen = torch.Generator().manual_seed(seed)
    o = OracleSF(S, A, D, tuple(hidden), tuple(acts), tsf_dim=tsf_dim)
    for _ in range(N):
        o.add_random_policy(gen)
    return o, gen


def build(o, precision, N, hidden=(256, 256), acts=('relu', 'relu'), **kw):
    meta = dict(S=o.S, A=o.A, D=o.D, hidden=list(hidden), acts=list(acts), N=N)
    return gu.build_g2(meta, oracle=o, hyper=hyper(precision, **kw))


def torch_dx(o, pols, x, Gs, emulate_bf16=False):
    """dL/dx of L = sum_p <psi_p(x), G_p> by torch autograd on the CPU: float64, or float32 with bf16-rounded operands (x, every
    W and the stored activations, straight-through) for the bf16 mode."""
    rb = _rb if emulate_bf16 else (lambda v: v)
    dt = torch.float32 if emulate_bf16 else torch.float64
    xr = x.detach().to(dt).clone().requires_grad_(True)
    loss = 0.0
    for p, G in zip(pols, Gs):
        h = rb(xr)
        for l, ((W, b), a) in enumerate(zip(o.psi[p], o.acts)):
            h = act_fn(a)(torch.addmm(b.to(dt), h, rb(W.to(dt)).t()))
            if l < len(o.acts) - 1:
                h = rb(h)
        loss = loss + (h.view(x.shape[0], o.A, o.D) * G.to(dt)).sum()
    loss.backward()
    return xr.grad


# ---- 1. dx against torch autograd ------------------------------------------------------------------------------------------------
CASES = [(4, 9, 12, 3, 1000, False), (4, 9, 12, 5, 33 * 128 - 5, False), (11, 27, 50, 2, 300, True), (4, 2, 20, 2, 32, False)]


@pytest.mark.parametrize('precision,tol', [('fp32', 2e-5), ('bf16', 1.5e-2), ('tf32x3', 2e-5), ('tf32', 6e-2)])
@pytest.mark.parametrize('S,A,D,N,B,hopper', CASES)
def test_state_gradient_vs_autograd(precision, tol, S, A, D, N, B, hopper):
    o, gen = make_oracle(S, A, D, N, seed=91)
    sf = build(o, precision, N, state_grad=True)
    x = synthetic_transitions(B, S, A, D, gen, hopper=hopper)[0]
    G = torch.randn(B, N, A, D, generator=gen) * 1e-4
    # No samples with an ambiguous ReLU gate (as the dense weight-gradient test does in tf32x3): there the float64 reference and
    # any fp32 evaluation may take different sides of the kink.  Measured on the CPU at B = 4219, N = 5: torch's own fp32 dx is
    # 2.1e-4 from the float64 one with them and 4.5e-7 without.
    if precision in ('fp32', 'tf32x3'):
        for p in range(N):
            G[relu_kink_rows(o, p, x), p] = 0.0
    bf = precision == 'bf16'
    # all policies through get_successors: dx sums over them
    xc = x.cuda().requires_grad_(True)
    (sf.get_successors(xc) * G.cuda()).sum().backward()
    ref = torch_dx(o, range(N), x, [G[:, p] for p in range(N)], emulate_bf16=bf)
    assert xc.grad.dtype == torch.float32 and xc.grad.shape == x.shape
    assert fro_err(xc.grad, ref) < tol, f'summed dx error {fro_err(xc.grad, ref)}'
    # one policy through get_successor and through the psi module
    for call in (lambda s: sf.get_successor(s, N - 1), lambda s: sf.psi[N - 1][0][0](s)):
        xc = x.cuda().requires_grad_(True)
        (call(xc) * G[:, N - 1].cuda()).sum().backward()
        ref = torch_dx(o, [N - 1], x, [G[:, N - 1]], emulate_bf16=bf)
        assert fro_err(xc.grad, ref) < tol, f'one-policy dx error {fro_err(xc.grad, ref)}'


def test_state_gradient_vs_autograd_tanh_cartpole_fp32():
    """Hidden width 32 (a reduction chunk narrower than one 256-wide stage), tanh hidden layers, fp32 mode."""
    S, A, D, N, B = 4, 2, 20, 3, 32
    o, gen = make_oracle(S, A, D, N, seed=13, hidden=(32, 32), acts=('tanh', 'tanh'))
    sf = build(o, 'fp32', N, hidden=(32, 32), acts=('tanh', 'tanh'), state_grad=True)
    x = synthetic_transitions(B, S, A, D, gen)[0]
    G = torch.randn(B, N, A, D, generator=gen)
    xc = x.cuda().requires_grad_(True)
    (sf.get_successors(xc) * G.cuda()).sum().backward()
    assert fro_err(xc.grad, torch_dx(o, range(N), x, [G[:, p] for p in range(N)])) < 2e-5
    xc = x.cuda().requires_grad_(True)
    (sf.psi[1][0][0](xc) * G[:, 1].cuda()).sum().backward()
    assert fro_err(xc.grad, torch_dx(o, [1], x, [G[:, 1]])) < 2e-5


def _tf32_rna(t):
    """fp32 -> nearest tf32, ties away from zero (cvt.rna.tf32.f32, the rounding of sfgpi_pack_f32)."""
    return ((t.float().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


@pytest.mark.parametrize('precision,S,K,n_pol,B', [
    ('fp32', 1, 50, 3, 77), ('fp32', 6, 256, 2, 1000), ('fp32', 20, 300, 2, 65), ('fp32', 100, 64, 3, 97),
    ('bf16', 4, 256, 5, 4219), ('bf16', 9, 256, 1, 33), ('bf16', 16, 256, 2, 500), ('bf16', 40, 256, 2, 300), ('bf16', 63, 256, 3, 129),
    ('tf32', 12, 256, 2, 200), ('tf32', 31, 256, 3, 64), ('tf32x3', 3, 256, 4, 1000), ('tf32x3', 13, 256, 2, 250),
    ('tf32x3', 31, 256, 1, 31),
])
def test_input_grad_kernel_vs_torch(precision, S, K, n_pol, B):
    """sfgpi_mlp_input_grad on its own, on random dZ0 in each mode's layout: every column block (4 .. 64, and several blocks for
    S > 64), hidden widths that are not multiples of the 256-wide chunk (fp32), ragged batches, a policy offset into the rows."""
    import ctypes as C
    from deep_successor_features_for_transfer_b200 import _lib
    from deep_successor_features_for_transfer_b200.library import NetSpec, _stream
    spec = NetSpec([S, K, K, 20], ['none', 'relu', 'none'], 2, 10)
    gen = torch.Generator().manual_seed(S * 1000 + K)
    lo = 1
    rows = torch.randn(lo + n_pol, spec.row_stride, generator=gen)
    W0 = rows[lo:, spec.w_off[0]:spec.w_off[0] + K * S].view(n_pol, K, S).double()
    dz = torch.randn(n_pol, B, K, generator=gen)
    g = _lib.InputGradArgs()
    g.net, g.precision, g.policy_lo, g.n_pol, g.B = spec.desc(), _lib.PREC[precision], lo, n_pol, B
    if precision == 'bf16':
        dz_dev, dzr, Wr = dz.bfloat16().cuda(), dz.bfloat16().double(), W0.float().bfloat16().double()
    elif precision == 'tf32x3':
        hi = _tf32_rna(dz)
        lo_part = _tf32_rna(dz - hi)
        dz_dev = torch.stack([hi, torch.zeros_like(hi), lo_part]).cuda()         # hi and lo slabs two slabs apart
        g.dz0_part_stride = 2 * n_pol * B * K
        dzr, Wr = hi.double() + lo_part.double(), W0
    else:
        dz_dev, dzr = dz.cuda(), dz.double()
        Wr = _tf32_rna(W0.float()).double() if precision == 'tf32' else W0
    params, dx = rows.cuda(), torch.full((B, S), float('nan'), device='cuda')
    g.params, g.dz0, g.dx = params.data_ptr(), dz_dev.data_ptr(), dx.data_ptr()
    assert _lib.lib().sfgpi_mlp_input_grad(C.byref(g), _stream()) == 0, _lib.lib().sfgpi_last_error()
    ref = torch.einsum('pbk,pks->bs', dzr, Wr)
    assert fro_err(dx, ref) < 1e-5, fro_err(dx, ref)
    dx2 = torch.empty_like(dx)
    g.dx = dx2.data_ptr()
    assert _lib.lib().sfgpi_mlp_input_grad(C.byref(g), _stream()) == 0
    assert torch.equal(dx, dx2)


# ---- 2. nothing else changes; 3. deterministic ----------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', PRECISIONS)
def test_state_gradient_changes_nothing_else_and_is_deterministic(precision):
    S, A, D, N, B = 4, 9, 12, 3, 33 * 128 - 5
    o, gen = make_oracle(S, A, D, N, seed=17)
    sg = build(o, precision, N, state_grad=True)
    plain = build(o, precision, N)
    x = synthetic_transitions(B, S, A, D, gen)[0].cuda()
    G = (torch.randn(B, N, A, D, generator=gen) * 1e-4).cuda()
    lib = sg._library
    xr = x.clone().requires_grad_(True)
    psi = sg.get_successors(xr)
    assert torch.equal(psi.detach(), lib.forward_psi(x))
    (psi * G).sum().backward()
    (plain.get_successors(x) * G).sum().backward()                 # no state gradient: same weight gradient, bit for bit
    assert torch.equal(lib.online.grad, plain._library.online.grad)
    dx1 = xr.grad.clone()
    for k in range(N):
        sg.psi[k][0][2].zero_grad()
    (sg.get_successors(x) * G).sum().backward()                    # the same library with detached states
    assert torch.equal(lib.online.grad, plain._library.online.grad)
    xr.grad = None
    (sg.get_successors(xr) * G).sum().backward()                   # a second identical backward: the same dx bits
    assert torch.equal(xr.grad, dx1)


# ---- 4. shape and dtype ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_state_gradient_keeps_dtype_and_shape(precision):
    S, A, D, N = 4, 9, 12, 2
    o, gen = make_oracle(S, A, D, N, seed=23)
    sf = build(o, precision, N, state_grad=True)
    s = torch.randn(S, generator=gen, dtype=torch.float64)
    G = torch.randn(1, A, D, generator=gen).cuda()
    x32 = s.float().cuda()[None].requires_grad_(True)              # the batch-1 call of the agents: get_successor(s[None])
    (sf.get_successor(x32, 1) * G).sum().backward()
    assert x32.grad.shape == (1, S) and x32.grad.dtype == torch.float32
    for dev in ('cuda', 'cpu'):
        s1 = s.to(dev).clone().requires_grad_(True)                # 1-D float64 state, on the device or on the host
        (sf.get_successor(s1, 1) * G).sum().backward()
        assert s1.grad.shape == (S,) and s1.grad.dtype == torch.float64 and s1.grad.device.type == dev
        assert torch.equal(s1.grad.cpu(), x32.grad[0].double().cpu())
    ref = torch_dx(o, [1], s.float()[None], [G.cpu()], emulate_bf16=precision == 'bf16')
    assert fro_err(x32.grad, ref) < (1.5e-2 if precision == 'bf16' else 2e-5)


# ---- 5. a learned encoder in front of psi, end to end ------------------------------------------------------------------------
def cpu_psi(o, i, hidden=(256, 256), acts=('relu', 'relu')):
    m = gu.model_lambda(list(hidden), list(acts))(o.S, o.A * o.D, (o.A, o.D), 1)[0]
    with torch.no_grad():
        for lin, (W, b) in zip(gu.linears(m), o.psi[i]):
            lin.weight.copy_(W)
            lin.bias.copy_(b)
    return m


def cpu_sf(o, N, gpu_sf):
    """The packed library's G2 state as plain CPU torch modules: psi / target nets, fit_w, and one torch.optim.Adam per policy
    over the same groups and learning rates, with the sf-like surface eager_g2_update / eager_g3_update use."""
    sf = types.SimpleNamespace(psi=[], fit_w=[], updates_since_target_updated=[0] * N, target_update_ev=gpu_sf.target_update_ev)
    for i in range(N):
        fw = torch.nn.Linear(o.D, 1, bias=False)
        with torch.no_grad():
            fw.weight.copy_(gpu_sf.fit_w[i].weight.detach().cpu())
        model, target = cpu_psi(o, i), cpu_psi(o, i)
        sf.fit_w.append(fw)
        sf.psi.append([[model, None, None], (target, None, None)])

    def GPI(next_states, i):
        w = sf.fit_w[i].weight.reshape(-1)
        return torch.stack([sf.psi[j][0][0](next_states) @ w for j in range(N)], dim=1), None
    sf.GPI = GPI
    return sf


def adam_like(gpu_optim, cpu_groups):
    return torch.optim.Adam([dict(params=p, lr=g['lr'], weight_decay=g['weight_decay']) for g, p in zip(gpu_optim.param_groups, cpu_groups)],
                            betas=(0.9, 0.999), eps=1e-8)


def encoder(S, seed):
    torch.manual_seed(seed)
    return torch.nn.Sequential(torch.nn.Linear(6, S), torch.nn.Tanh())


def encoded_batch(enc, raw, raw_next, rest):
    actions, rs, phis, gammas = rest
    states = enc(raw)
    with torch.no_grad():
        next_states = enc(raw_next)
    return states, actions, rs, phis, next_states, gammas


def test_learned_encoder_g2_steps_match_cpu_torch():
    S, A, D, N, B, i, K = 4, 9, 12, 3, 256, 1, 3
    o, gen = make_oracle(S, A, D, N, seed=31)
    sf = build(o, 'fp32', N, state_grad=True)
    ref = cpu_sf(o, N, sf)
    ref.psi[i][0][2] = adam_like(sf.psi[i][0][2], [list(ref.psi[i][0][0].parameters()), list(ref.fit_w[i].parameters())])
    enc_c = encoder(S, 5)
    enc_g = copy.deepcopy(enc_c).cuda()
    opt_c, opt_g = torch.optim.Adam(enc_c.parameters(), lr=1e-3), torch.optim.Adam(enc_g.parameters(), lr=1e-3)
    enc0 = enc_c[0].weight.detach().clone()
    for k in range(K):
        raw, raw_next = torch.randn(B, 6, generator=gen), torch.randn(B, 6, generator=gen)
        _, actions, rs, phis, _, gammas = synthetic_transitions(B, S, A, D, gen)
        rest = (actions, rs, phis, gammas)
        opt_g.zero_grad()
        got = eager_g2_update(sf, encoded_batch(enc_g, raw.cuda(), raw_next.cuda(), tuple(v.cuda() for v in rest)), i, True)
        opt_g.step()
        opt_c.zero_grad()
        want = eager_g2_update(ref, encoded_batch(enc_c, raw, raw_next, rest), i, True)
        opt_c.step()
        assert np.allclose([float(v) for v in got], [float(v) for v in want], rtol=2e-5, atol=1e-8), (k, got, want)
    for (W, b), lin in zip(gu.psi_params(sf, i), gu.linears(ref.psi[i][0][0])):
        assert rel_err(W, lin.weight.detach()) < STEP_TOL and rel_err(b, lin.bias.detach()) < STEP_TOL
    assert rel_err(sf.fit_w[i].weight.detach().cpu(), ref.fit_w[i].weight.detach()) < STEP_TOL
    for pg, pc in zip(enc_g.parameters(), enc_c.parameters()):
        assert rel_err(pg.detach().cpu(), pc.detach()) < STEP_TOL
    assert not torch.equal(enc_c[0].weight.detach(), enc0)         # the encoder did learn from the psi loss


def test_learned_encoder_feeding_psi_and_g_matches_cpu_torch():
    """G3: the encoder feeds psi AND the TSF g function; one backward's encoder gradient through both paths."""
    S, A, D, N, B, i, Gd = 4, 9, 12, 3, 256, 2, 100
    o, gen = make_oracle(S, A, D, N, seed=37, tsf_dim=Gd)
    from deep_successor_features_for_transfer_b200.tsfdqn import DeepTSF, TSFDQN, ReplayBuffer
    hp = hyper('fp32', state_grad=True, g_h_function_dims=Gd, beta_loss_coefficient=1.0)
    dsf = DeepTSF(pytorch_model_handle=gu.model_lambda([256, 256], ['relu', 'relu']), target_update_ev=1000, hyperparameters=hp)
    ag = TSFDQN(deep_sf=dsf, buffer_handle=lambda: ReplayBuffer(), gamma=0.9, T=500, encoding=None, use_gpi=True, hyperparameters=hp)
    ag.reset()
    for k in range(N):
        ag.add_training_task(gu.FakeTask(S, A, D, k))
    ref_sf = cpu_sf(o, N, dsf)
    g_c = [torch.nn.Linear(S, Gd) for _ in range(N)]
    h_c = torch.nn.Linear(Gd, D)
    with torch.no_grad():
        for k in range(N):
            gu.load_policy(dsf, k, o.psi[k], o.w[k])
            ref_sf.fit_w[k].weight.copy_(o.w[k].reshape(1, -1))
            for lin_g, lin_c, (W, b) in ((ag.g_functions[k], g_c[k], o.g[k]),):
                lin_g.weight.data.copy_(W)
                lin_g.bias.data.copy_(b)
                lin_c.weight.copy_(W)
                lin_c.bias.copy_(b)
        ag.h_function.weight.data.copy_(o.h[0])
        ag.h_function.bias.data.copy_(o.h[1])
        h_c.weight.copy_(o.h[0])
        h_c.bias.copy_(o.h[1])
    ref_sf.psi[i][0][2] = torch.optim.Adam([p for m in (ref_sf.psi[i][0][0], ref_sf.fit_w[i], g_c[i], h_c) for p in m.parameters()])
    ref = types.SimpleNamespace(sf=ref_sf, g_functions=g_c, h_function=h_c, hyperparameters=dict(beta_loss_coefficient=1.0))
    enc_c = encoder(S, 7)
    enc_g = copy.deepcopy(enc_c).cuda()
    raw, raw_next = torch.randn(B, 6, generator=gen), torch.randn(B, 6, generator=gen)
    _, actions, rs, phis, _, gammas = synthetic_transitions(B, S, A, D, gen)
    rest = (actions, rs, phis, gammas)
    got = eager_g3_update(ag, encoded_batch(enc_g, raw.cuda(), raw_next.cuda(), tuple(v.cuda() for v in rest)), i, True)
    want = eager_g3_update(ref, encoded_batch(enc_c, raw, raw_next, rest), i, True)
    assert np.allclose([float(v) for v in got], [float(v) for v in want], rtol=2e-5, atol=1e-8)
    for pg, pc in zip(enc_g.parameters(), enc_c.parameters()):
        assert pc.grad is not None and pc.grad.abs().max() > 0
        assert fro_err(pg.grad, pc.grad) < 2e-5, fro_err(pg.grad, pc.grad)


# ---- 6. errors ------------------------------------------------------------------------------------------------------------------
def test_state_gradient_errors():
    from deep_successor_features_for_transfer_b200.library import PackedSFLibrary
    from deep_successor_features_for_transfer_b200.sfdqn import DeepSF
    with pytest.raises(ValueError, match='autograd'):
        PackedSFLibrary(state_grad=True)
    with pytest.raises(ValueError, match='autograd'):
        DeepSF(pytorch_model_handle=gu.model_lambda([256, 256], ['relu', 'relu']), hyperparameters=dict(gu.HYPER, state_grad=True))
    S, A, D, N, B = 4, 9, 12, 3, 256
    o, gen = make_oracle(S, A, D, N, seed=41)
    sf = build(o, 'fp32', N, state_grad=True)
    lib = sf._library
    tr = gu.cuda_tr(synthetic_transitions(B, S, A, D, gen))
    x = tr[0].clone().requires_grad_(True)
    target = sf.psi[1][1][0]
    with pytest.raises(RuntimeError, match='no_grad'):             # target nets are constants
        target(x)
    with torch.no_grad():
        assert torch.equal(target(x), lib.forward_psi(tr[0], 1, 1, target=True)[:, 0])
    assert torch.equal(target(x.detach()), lib.forward_psi(tr[0], 1, 1, target=True)[:, 0])
    model = sf.psi[1][0][0]
    psi = model(x)
    d_psi = torch.ones_like(psi, requires_grad=True)
    with pytest.raises(RuntimeError):                              # no double backward
        torch.autograd.grad(psi, [lib.online, x], d_psi, create_graph=True)[1].sum().backward()
    psi = model(x)
    sf.update_successor(tr, 1, True)                               # the fused step moves the online rows
    with pytest.raises(RuntimeError):
        psi.sum().backward()
    lib.shard = types.SimpleNamespace(world=2)
    with pytest.raises(NotImplementedError):
        lib.psi(x, 0, 1)
    lib.shard = None
    model(x).sum().backward()                                      # and the library still works
    assert x.grad is not None and x.grad.abs().max() > 0
