"""
-m gpu: every precision mode at the psi net shapes the rest of the suite never builds, against a float64 reference written here.

The other tensor-core tests all use [S, 256, 256, 256, A*D] with activations [none, relu, relu, none] and S = 4 or 11.  The
kernels hold logic that depends on the depth, the activation of each layer and the state width; each architecture below is the
only one in the suite that reaches some of it:

  L3      Linear x 3, one ReLU hidden layer (Reacher)   Lh = L - 2 = 1: the output layer drains TMEM accumulator 0, one-item dgrad
                                                        chain, the smallest operand shadow
  L5tanh  Linear x 5, three Tanh hidden layers (Hopper) odd Lh, no ReLU anywhere (mask-free backward, tf32 relu = false), the tanh
                                                        forward epilogue and derivative in every mode, 6 output chunks
  L8      Linear x 8, six ReLU hidden layers (Hopper)   the deepest net: (1 + 6) * 256 + 1350 = 3142 > 3072 bias floats, so the
                                                        chain kernel keeps its biases single-buffered
  mixed   ReLU after layer 0, a linear hidden layer,    an activation on the first layer (its ReLU mask and the state gradient
          then tanh and relu (Reacher)                  through it), relu / tanh / none interleaved
  S17     headline net, S = 17                          bf16 first layer over 2 k-steps (tf32: 3)
  S31     headline net, S = 31                          the tf32 / tf32x3 limit (4 k-steps of 8)
  S63     headline net, S = 63 (bf16 and fp32 only)     the bf16 limit: 4 k-steps of 16, xo = [x | 1] fills its 64 columns

each at two launch sizes: 'chain' (N = 3, B = 333: 9 row tiles, a ragged last one; the layer-pipelined chain kernel) and 'pair'
(N = 2, B = 75 * 128 + 7: 152 row tiles > 148 SMs; the ping-pong pair kernel and, in bf16, the paired dgrad mode).

Per case: psi of the online and target nets; GPI q, action and task for one reward vector and for 13 (blocked column order,
padding); the weight gradients of every layer and dL/dx from one dense dL/dpsi backward (state_grad=True); one fused train
step with GPI (losses, post-step weights, Adam's first moment m = 0.1 g).  Two references, both float64, both built from the
library's own weights:
  exact     plain float64 arithmetic: the mode's stated tolerance (fp32 / tf32x3: the fp32 parity bounds; bf16: BF16_TOL 2e-2;
            tf32: 2e-3 on psi / q);
  emulated  (bf16, tf32) float64 arithmetic with the operands of every GEMM -- states, weights, stored activations, dZ, the
            folded GPI weights -- rounded to the mode's type where the kernels round them: a tight bound, so that a wrong bias
            or derivative at one deep layer cannot hide inside 2e-2.
Every bound is set from the reference's own float32-versus-float64 spread on the CPU (the same computation in float32
against float64, at every case of the matrix: TIGHT below), never from kernel output.
"""
import types
import zlib

import pytest
import torch
import torch.nn.functional as F

from deep_successor_features_for_transfer_b200 import workloads as wl
from oracle.sf_oracle import act_fn
from tests import gpu_util as gu
from tests.golden_util import rel_err
from tests.test_gpu_tf32 import MOMENT_TOL, check_moments, relu_kink_rows, weights_close

pytestmark = pytest.mark.gpu

REACHER, HOPPER = wl.ENVS['reacher'], wl.ENVS['hopper']
HEADLINE = dict(hidden=[256, 256], acts=['relu', 'relu'])
ALL = ('fp32', 'bf16', 'tf32', 'tf32x3')
ARCHS = {
    'L3': dict(env=REACHER, hidden=[256], acts=['relu'], precisions=ALL),
    'L5tanh': dict(env=HOPPER, hidden=[256] * 3, acts=['tanh'] * 3, precisions=ALL),
    'L8': dict(env=HOPPER, hidden=[256] * 6, acts=['relu'] * 6, precisions=ALL),
    'mixed': dict(env=REACHER, custom=True, precisions=ALL),
    'S17': dict(env=dict(S=17, A=9, D=12), **HEADLINE, precisions=ALL),
    'S31': dict(env=dict(S=31, A=9, D=12), **HEADLINE, precisions=ALL),
    'S63': dict(env=dict(S=63, A=9, D=12), **HEADLINE, precisions=('fp32', 'bf16')),
}
BATCHES = {'chain': (3, 333), 'pair': (2, 75 * 128 + 7)}
NW = 13                     # reward vectors of the multi-vector GPI: one full block of 8 and a padded one of 5
SEED = 1234

# Stated tolerances against the exact reference (include/sfgpi.h, PackedSFLibrary.set_precision, tests/test_gpu_bf16.py,
# tests/test_gpu_tf32.py, tests/test_gpu_autograd.py).  fwd: psi / q / GPI key values, scale-relative; grad: dW, db, dx, relative
# Frobenius (ReLU-kink samples removed from dL/dpsi in every mode); loss: relative error of (loss, l1, l2) of the train step;
# m: Adam's first moment after the step (0.1 g), relative Frobenius per layer (fp32 / tf32x3: check_moments' bounds); tie: a
# state whose GPI top-1 / top-2 q are within tie * max|q| may take the other a' in the step, which moves the losses by up to
# ~4 / B and m by ~2 / B (bf16 / tf32 against the exact reference: no allowance, the stated bounds hold without it).
# The float32 evaluation of the exact reference stays within 8.8e-7 (psi, q), 7.7e-7 (grad), 1.5e-7 (loss), 2.9e-7 (m of the
# output layer) and 3.6e-4 (m of a hidden layer, after a flipped ReLU gate) of its float64 evaluation over the whole matrix.
# bf16 gradients are not held against the exact reference: the emulated reference itself is up to 1.1e-1 from it (L8: ReLU
# gates flipped by bf16 rounding), as in the existing bf16 backward tests, which hold them against the emulation only.
STATED = {
    'fp32': dict(fwd=1e-5, grad=2e-5, loss=2e-5, tie=1e-5),
    'tf32x3': dict(fwd=1e-5, grad=2e-5, loss=2e-5, tie=1e-5),
    'bf16': dict(fwd=2e-2, fro=1e-2, grad=None, loss=3e-2, m=9e-2, tie=0.0),
    'tf32': dict(fwd=2e-3, grad=6e-2, loss=2e-3, m=6e-2, tie=0.0),
}
# Against the emulated reference (bf16, tf32), all relative Frobenius: about 4x the largest float32-versus-float64 spread of
# that reference over the matrix on the CPU (in brackets; the worst case named):
#   bf16  fwd 6e-4 [1.3e-4 L5tanh-chain]   grad 2e-2 [5.6e-3 mixed-chain]   loss 1e-5 [2.5e-7 without an a' flip]   m 5e-3
#         [1.2e-3 mixed-chain; 3.1e-3 with an a' flip, L5tanh-chain]   tie 5e-3 [q, max element: 2.3e-3]
#   tf32  fwd 3e-4 [7.5e-5 L5tanh-pair]    grad 4e-2 [1.0e-2 L8-chain]      loss 2e-6 [3.5e-7 mixed-pair]           m 4e-3
#         [9.5e-4 S17-pair]                tie 1e-3 [q, max element: 3.8e-4]
# For scale, the emulated reference's own distance to the exact one (the mode's intrinsic error): bf16 fwd 4.3e-3, grad 1.1e-1,
# loss 3.8e-4, m 7.2e-2; tf32 fwd 5.7e-4, grad 3.6e-2, loss 2.3e-5, m 2.7e-2.
# tf32x3 gradients: the tensor cores' fp32 accumulation error grows with the length of the reductions (tests/test_gpu_autograd.py:
# 1.1e-5 at B = 4219, 1.3e-5 with Hopper's 1350 output columns) and with the number of chained GEMMs between the loss and a
# layer's gradient (L - 1 for layer 0; 3 in the 4-layer net the 2e-5 bound was set on).  So the bound scales with both:
# 2e-5 * max(1, B / 4219) * max(1, (L - 1) / 3).  Measured on B200 (1000 W), layer 0's dW: L5tanh pair 3.4e-5 (bound 6.1e-5),
# L8 chain 2.0e-5 (4.7e-5), L8 pair 4.9e-5 (1.1e-4); the psi / q / loss bounds hold unscaled.
TF32X3_GRAD_B, TF32X3_GRAD_GEMMS = 4219, 3
TIGHT = {
    'bf16': dict(fwd=6e-4, grad=2e-2, loss=1e-5, m=5e-3, tie=5e-3),
    'tf32': dict(fwd=3e-4, grad=4e-2, loss=2e-6, m=4e-3, tie=1e-3),
}


# ---- building the libraries ------------------------------------------------------------------------------------------------
def mixed_model(num_inputs, output_dim, reshape_dim, reshape_axis=1):
    """A psi net model_lambda cannot express: ReLU after the input layer, a linear hidden layer, then tanh and relu."""
    m = torch.nn.Sequential(torch.nn.Linear(num_inputs, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256),
                            torch.nn.Linear(256, 256), torch.nn.Tanh(), torch.nn.Linear(256, 256), torch.nn.ReLU(),
                            torch.nn.Linear(256, output_dim), torch.nn.Unflatten(reshape_axis, reshape_dim))
    return m, torch.nn.MSELoss(), None


def build(arch, precision, N):
    """workloads.build_sf_library's DeepSF with autograd and state_grad on: the same seeded weights in every precision mode."""
    from deep_successor_features_for_transfer_b200.sfdqn import DeepSF
    c = ARCHS[arch]
    env = c['env']
    handle = mixed_model if c.get('custom') else wl.model_lambda(c['hidden'], c['acts'])
    sf = DeepSF(pytorch_model_handle=handle, target_update_ev=1000,
                hyperparameters=dict(wl.HYPER, precision=precision, autograd=True, state_grad=True))
    sf.reset()
    for k in range(N):
        with wl.seeded_policy_init(SEED + k):
            sf.add_training_task(wl.ShapeTask(env['S'], env['A'], env['D'], k))
    assert sf._library.precision == precision
    return sf


def net_of(sf, N):
    """The library's weights as float64 CPU tensors: online / target layers and reward vectors of every policy."""
    spec = sf._library.spec
    return types.SimpleNamespace(
        acts=list(spec.acts), A=spec.n_actions, D=spec.n_features,
        psi=[[(W.double(), b.double()) for W, b in gu.psi_params(sf, i)] for i in range(N)],
        tgt=[[(W.double(), b.double()) for W, b in gu.psi_params(sf, i, target=True)] for i in range(N)],
        w=[sf.fit_w[i].weight.detach().cpu().double().reshape(-1) for i in range(N)])


def inputs(arch, batch):
    c = ARCHS[arch]
    S, A, D = c['env']['S'], c['env']['A'], c['env']['D']
    N, B = BATCHES[batch]
    gen = torch.Generator().manual_seed(zlib.crc32(f'{arch}-{batch}'.encode()))
    tr = wl.synthetic_transitions(B, S, A, D, gen, hopper=c['env'] is HOPPER)
    G = torch.randn(B, N, A, D, generator=gen) * 1e-4
    w13 = torch.rand(NW, D, generator=gen) * 0.02 - 0.01
    return tr, G, w13


# ---- the float64 reference ---------------------------------------------------------------------------------------------------
def _tf32_rna(t):
    """fp32 -> nearest tf32, ties away from zero (cvt.rna.tf32.f32)."""
    return ((t.float().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


ROUND = {'bf16': lambda t: t.float().bfloat16().to(t.dtype), 'tf32': lambda t: _tf32_rna(t).to(t.dtype)}


class _RoundGrad(torch.autograd.Function):
    """Identity forward; the backward rounds dZ, an operand of the dgrad chain and of wgrad."""

    @staticmethod
    def forward(ctx, t, mode):
        ctx.mode = mode
        return t.view_as(t)

    @staticmethod
    def backward(ctx, g):
        return ROUND[ctx.mode](g), None


def _op(t, mode):
    """Straight-through operand rounding: the value the tensor core consumes, the full-precision gradient path."""
    return t if mode is None else t + (ROUND[mode](t) - t).detach()


def mlp(layers, acts, x, mode=None):
    """psi = the net at x -> (output [B, A*D], input of the output layer [B, 256]).  mode: None (exact) or the rounding points
    of the 'bf16' / 'tf32' kernels."""
    h = _op(x, mode)
    for l, ((W, b), a) in enumerate(zip(layers, acts)):
        z = torch.addmm(b, h, _op(W, mode).t())
        if mode is not None:
            z = _RoundGrad.apply(z, mode)
        if l == len(layers) - 1:
            return z, h
        h = _op(act_fn(a)(z), mode)


def gpi_q(net, layers_of, x, w, mode=None):
    """q [B, N, A] for reward vector w: psi . w, or (emulated) the kernels' folded form q = h . round(Wq)^T + bq."""
    qs = []
    for layers in layers_of:
        out, h = mlp(layers, net.acts, x, mode)
        if mode is None:
            qs.append(out.view(-1, net.A, net.D) @ w)
        else:
            Wo, bo = layers[-1]
            Wq = torch.einsum('d,adk->ak', w, Wo.view(net.A, net.D, -1))
            qs.append(torch.addmm(bo.view(net.A, net.D) @ w, h, ROUND[mode](Wq).t()))
    return torch.stack(qs, dim=1)


def reference(net, tr, G, w13, dt=torch.float64, mode=None):
    """Every quantity the tests compare, in dtype dt (float64; float32 only for the spread study)."""
    cv = lambda t: t.to(dt)
    net = types.SimpleNamespace(acts=net.acts, A=net.A, D=net.D, psi=[[(cv(W), cv(b)) for W, b in L] for L in net.psi],
                                tgt=[[(cv(W), cv(b)) for W, b in L] for L in net.tgt], w=[cv(w) for w in net.w])
    states, actions, rs, phis, next_states, gammas = tr
    x, G, w13 = cv(states), cv(G), cv(w13)
    N, B = len(net.psi), x.shape[0]
    r = {}
    with torch.no_grad():
        r['psi'] = torch.stack([mlp(L, net.acts, x, mode)[0].view(B, net.A, net.D) for L in net.psi], dim=1)
        r['psi_t'] = torch.stack([mlp(L, net.acts, x, mode)[0].view(B, net.A, net.D) for L in net.tgt], dim=1)
        r['q1'] = gpi_q(net, net.psi, x, net.w[N - 1], mode)
        r['q13'] = torch.stack([gpi_q(net, net.psi, x, w13[k], mode) for k in range(NW)])
    # one dense backward over all policies: dW, db of every layer and dL/dx
    xr = x.clone().requires_grad_(True)
    leaves = [[(W.clone().requires_grad_(True), b.clone().requires_grad_(True)) for W, b in L] for L in net.psi]
    loss = sum((mlp(L, net.acts, xr, mode)[0].view(B, net.A, net.D) * G[:, p]).sum() for p, L in enumerate(leaves))
    loss.backward()
    r['grads'] = [[(W.grad, b.grad) for W, b in L] for L in leaves]
    r['dx'] = xr.grad
    r['step'] = train_step_ref(net, [cv(t) if t.is_floating_point() else t for t in tr], N - 1, mode)
    return r


def train_step_ref(net, tr, i, mode=None, lr=1e-3):
    """The G2 update of policy i with GPI (sfdqn.py:303-371) and one fresh Adam step: losses, post-step weights, m = 0.1 g."""
    states, actions, rs, phis, next_states, gammas = tr
    B = states.shape[0]
    idx = torch.arange(B)
    with torch.no_grad():
        q = gpi_q(net, net.psi, next_states, net.w[i], mode)
        top2 = q.reshape(B, -1).topk(2, dim=1).values
        next_a = torch.argmax(q.max(dim=1).values, dim=-1)
        targets = phis + gammas[:, None] * mlp(net.tgt[i], net.acts, next_states, mode)[0].view(B, net.A, net.D)[idx, next_a]
    leaves = [(W.clone().requires_grad_(True), b.clone().requires_grad_(True)) for W, b in net.psi[i]]
    w = net.w[i].clone().requires_grad_(True)
    cur = mlp(leaves, net.acts, states, mode)[0].view(B, net.A, net.D)
    merge = cur.clone()
    merge[idx, actions] = targets
    l1 = F.mse_loss(cur, merge)
    l2 = F.mse_loss(phis @ w[:, None], rs)
    (l1 + l2).backward()
    adam = lambda p, g: p.detach() - lr * g / (g.abs() + 1e-8)        # torch.optim.Adam's first step, no weight decay
    return dict(losses=torch.stack([l1 + l2, l1, l2]).detach(),
                post=[(adam(W, W.grad), adam(b, b.grad)) for W, b in leaves], m=[0.1 * W.grad for W, _ in leaves],
                w=adam(w, w.grad), gap=(top2[:, 0] - top2[:, 1]) / q.abs().max())


def ties(step, band):
    """States whose GPI top-1 / top-2 q are within band of the scale: a kernel inside that band may take the other a'."""
    return int((step['gap'] < band).sum())


_CACHE = {}


def cached_reference(arch, batch, net, mode):
    """(transitions, dL/dpsi, 13 reward vectors, reference) of one architecture and batch, computed once for all modes."""
    key = (arch, batch, mode)
    if key in _CACHE:
        assert all(torch.equal(W, W0) for L, L0 in zip(net.psi, _CACHE[key][4].psi) for (W, _), (W0, _) in zip(L, L0))
    else:
        tr, G, w13 = inputs(arch, batch)
        o = types.SimpleNamespace(psi=[[(W.float(), b.float()) for W, b in L] for L in net.psi], acts=net.acts)
        for p in range(G.shape[1]):           # no samples with an ambiguous ReLU gate in dL/dpsi (tests/test_gpu_tf32.py)
            G[relu_kink_rows(o, p, tr[0]), p] = 0.0
        _CACHE[key] = (tr, G, w13, reference(net, tr, G, w13, mode=mode), net)
    return _CACHE[key][:4]


def fro_err(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


# ---- the test -----------------------------------------------------------------------------------------------------------------
CASES = [pytest.param(arch, prec, batch, id=f'{arch}-{prec}-{batch}')
         for arch, c in ARCHS.items() for prec in c['precisions'] for batch in BATCHES]


@pytest.mark.parametrize('arch,precision,batch', CASES)
def test_architecture_vs_float64(arch, precision, batch):
    from deep_successor_features_for_transfer_b200 import _lib
    from deep_successor_features_for_transfer_b200.library import _stream
    N, B = BATCHES[batch]
    sf = build(arch, precision, N)
    lib = sf._library
    net = net_of(sf, N)
    tr, G, w13, ex = cached_reference(arch, batch, net, None)
    em = cached_reference(arch, batch, net, precision)[3] if precision in TIGHT else None
    st, tt = dict(STATED[precision]), TIGHT.get(precision)
    if precision == 'tf32x3':
        st['grad'] *= max(1.0, B / TF32X3_GRAD_B) * max(1.0, (len(lib.spec.acts) - 1) / TF32X3_GRAD_GEMMS)
    x = tr[0].cuda()
    msg = f'{arch} {precision} {batch}'

    # 1. forward: psi of the online and the target nets
    psi = sf.get_successors(x).detach().cpu()
    psi_t = lib.forward_psi(x, 0, N, target=True).cpu()
    assert rel_err(psi, ex['psi']) < st['fwd'] and rel_err(psi_t, ex['psi_t']) < st['fwd'], (msg, rel_err(psi, ex['psi']))
    if 'fro' in st:
        assert fro_err(psi, ex['psi']) < st['fro'], msg
    if em is not None:
        assert fro_err(psi, em['psi']) < tt['fwd'] and fro_err(psi_t, em['psi_t']) < tt['fwd'], (msg, fro_err(psi, em['psi']))

    # 2. GPI, one reward vector (policy N-1's w) over every policy, and 13 vectors in one launch
    q_ref = ex['q1']
    q, task = sf.GPI(x, N - 1)
    assert rel_err(q.cpu(), q_ref) < st['fwd'], (msg, rel_err(q.cpu(), q_ref))
    if em is not None:
        assert fro_err(q.cpu(), em['q1']) < tt['fwd'], (msg, fro_err(q.cpu(), em['q1']))
    ok, nbad = gu.argmax_mismatch_ok(q_ref, q_ref.max(dim=2).values.argmax(dim=1), task.cpu(), 'task', st['fwd'])
    assert ok, f'{msg}: {nbad} task mismatches outside tolerance'
    _, key_a, _ = lib.gpi(x, sf.fit_w[N - 1].weight, want_q=False)
    act, val = lib.decode_keys(key_a, want_value=True)
    ok, nbad = gu.argmax_mismatch_ok(q_ref, q_ref.max(dim=1).values.argmax(dim=-1), act.cpu(), 'action', st['fwd'])
    assert ok, f'{msg}: {nbad} action mismatches outside tolerance'
    assert torch.equal(val, q.reshape(B, -1).max(dim=1).values)                     # the keys carry the q the kernel returned

    ka = torch.empty(NW, B, dtype=torch.int64, device='cuda')
    kt = torch.empty(NW, B, dtype=torch.int64, device='cuda')
    _lib.call('sfgpi_keys_fill', ka.data_ptr(), ka.numel(), _stream())
    _lib.call('sfgpi_keys_fill', kt.data_ptr(), kt.numel(), _stream())
    wd = w13.cuda().contiguous()
    a = lib._fwd_args(lib.online, 0, N, x)
    a.w, a.n_w, a.w_diag, a.task_base = wd.data_ptr(), NW, 0, 0
    a.key_action, a.key_task = ka.data_ptr(), kt.data_ptr()
    lib._forward(a, 'online')
    act13, val13 = lib.decode_keys(ka, want_value=True)
    task13 = lib.decode_keys(kt).cpu()
    act13, val13 = act13.cpu(), val13.cpu()
    for k in range(NW):
        qk = ex['q13'][k]
        scale = float(qk.abs().max())
        assert float((val13[k] - qk.reshape(B, -1).max(dim=1).values).abs().max()) < st['fwd'] * scale, (msg, k)
        if em is not None:
            ve = em['q13'][k].reshape(B, -1).max(dim=1).values
            assert fro_err(val13[k], ve) < tt['fwd'], (msg, k, fro_err(val13[k], ve))
        ok, nb = gu.argmax_mismatch_ok(qk, qk.max(dim=1).values.argmax(dim=-1), act13[k], 'action', st['fwd'])
        assert ok, f'{msg} vector {k}: {nb} action mismatches outside tolerance'
        ok, nb = gu.argmax_mismatch_ok(qk, qk.max(dim=2).values.argmax(dim=1), task13[k], 'task', st['fwd'])
        assert ok, f'{msg} vector {k}: {nb} task mismatches outside tolerance'

    # 3. + 4. one backward of a dense dL/dpsi over every policy: dW, db of every layer and dL/dx
    xc = x.clone().requires_grad_(True)
    (sf.get_successors(xc) * G.cuda()).sum().backward()
    for p in range(N):
        for l, lin in enumerate(gu.linears(sf.psi[p][0][0].net)):
            for got, name, j in ((lin.weight.grad, 'dW', 0), (lin.bias.grad, 'db', 1)):
                if st['grad'] is not None:
                    assert fro_err(got, ex['grads'][p][l][j]) < st['grad'], (msg, p, l, name, fro_err(got, ex['grads'][p][l][j]))
                if em is not None:
                    assert fro_err(got, em['grads'][p][l][j]) < tt['grad'], (msg, p, l, name, fro_err(got, em['grads'][p][l][j]))
    assert xc.grad.shape == x.shape
    if st['grad'] is not None:
        assert fro_err(xc.grad, ex['dx']) < st['grad'], (msg, 'dx', fro_err(xc.grad, ex['dx']))
    if em is not None:
        assert fro_err(xc.grad, em['dx']) < tt['grad'], (msg, 'dx', fro_err(xc.grad, em['dx']))

    # 5. one fused train step of policy N-1 with GPI
    i = N - 1
    m_before = lib.m[i].clone()
    losses = torch.stack([torch.as_tensor(float(v)) for v in sf.update_successor(gu.cuda_tr(tr), i, True)]).double()
    assert float(m_before.abs().max()) == 0.0
    ref = ex['step']
    loss_err = lambda r: float(((losses - r['losses']).abs() / r['losses'].abs()).max())
    assert loss_err(ref) < st['loss'] + 4.0 * ties(ref, st['tie']) / B, (msg, losses, ref['losses'])
    ms = [mW for mW, _ in lib.spec.views(lib.m[i].detach().cpu())]
    if precision in ('fp32', 'tf32x3'):
        for l, (W, b) in enumerate(gu.psi_params(sf, i)):
            assert weights_close(W, ref['post'][l][0]) and weights_close(b, ref['post'][l][1]), (msg, l)
        check_moments([(l, fro_err(ms[l], ref['m'][l])) for l in range(len(ms))], len(ms),
                      out_tol=MOMENT_TOL + 2.0 * ties(ref, st['tie']) / B)
        assert rel_err(sf.fit_w[i].weight.detach().cpu().reshape(-1), ref['w']) < 1e-4, msg
    else:
        e = em['step']
        e_ties = ties(e, tt['tie']) / B
        assert loss_err(e) < tt['loss'] + 4.0 * e_ties, (msg, losses, e['losses'])
        for l in range(len(ms)):
            assert fro_err(ms[l], ref['m'][l]) < st['m'], (msg, l, fro_err(ms[l], ref['m'][l]))
            assert fro_err(ms[l], e['m'][l]) < tt['m'] + 2.0 * e_ties, (msg, l, fro_err(ms[l], e['m'][l]))
