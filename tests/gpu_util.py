"""Helpers for the -m gpu parity tests: build the CUDA-side library from a golden fixture or from an OracleSF."""
from collections import OrderedDict

import torch

from tests.golden_util import n_layers, t

from deep_successor_features_for_transfer_b200.workloads import ACTS, HYPER, ShapeTask as FakeTask, model_lambda  # noqa: F401,E402
# (the shapes-only task, the mains' MLP factory and the cfg hyper-parameters live in the package: bench.py's measured arm uses
# them too and must not import test helpers)


def linears(m):
    return [x for x in m.modules() if isinstance(x, torch.nn.Linear)]


def load_policy(sf, i, layers, w, g=None):
    """Overwrite policy i's online+target nets, w (and g) with given CPU tensors, through the module views."""
    with torch.no_grad():
        for which in (0, 1):
            for lin, (W, b) in zip(linears(sf.psi[i][which][0].net), layers):
                lin.weight.data.copy_(W)
                lin.bias.data.copy_(b)
        fw = sf.fit_w[i]
        dst = fw.weight.data if isinstance(fw, torch.nn.Module) else fw
        dst.copy_(w.reshape(dst.shape))


def build_g2(meta, z=None, oracle=None, hyper=None):
    from deep_successor_features_for_transfer_b200.sfdqn import DeepSF
    sf = DeepSF(pytorch_model_handle=model_lambda(meta['hidden'], meta['acts']), use_true_reward=False,
                target_update_ev=meta.get('target_update_ev', 1000), hyperparameters=dict(hyper or HYPER))
    sf.reset()
    for i in range(meta['N']):
        sf.add_training_task(FakeTask(meta['S'], meta['A'], meta['D'], i))
    for i in range(meta['N']):
        if z is not None:
            layers = [(t(z[f'init.psi{i}.W{l}']), t(z[f'init.psi{i}.b{l}'])) for l in range(n_layers(meta))]
            load_policy(sf, i, layers, t(z[f'init.w{i}']))
        else:
            load_policy(sf, i, oracle.psi[i], oracle.w[i])
    return sf


def build_g3(meta, z=None, oracle=None):
    from deep_successor_features_for_transfer_b200.tsfdqn import DeepTSF, TSFDQN, ReplayBuffer
    hyper = dict(HYPER, g_h_function_dims=meta['gdim'], beta_loss_coefficient=meta['beta'])
    dsf = DeepTSF(pytorch_model_handle=model_lambda(meta['hidden'], meta['acts']), use_true_reward=False,
                  target_update_ev=meta.get('target_update_ev', 1000), hyperparameters=hyper)
    ag = TSFDQN(deep_sf=dsf, buffer_handle=lambda: ReplayBuffer(), gamma=0.9, T=500, encoding=None,
                use_gpi=meta.get('use_gpi', True), hyperparameters=hyper)
    ag.reset()
    for i in range(meta['N']):
        ag.add_training_task(FakeTask(meta['S'], meta['A'], meta['D'], i))
    with torch.no_grad():
        for i in range(meta['N']):
            if z is not None:
                layers = [(t(z[f'init.psi{i}.W{l}']), t(z[f'init.psi{i}.b{l}'])) for l in range(n_layers(meta))]
                load_policy(dsf, i, layers, t(z[f'init.w{i}']))
                gW, gb = t(z[f'init.g{i}.W']), t(z[f'init.g{i}.b'])
            else:
                load_policy(dsf, i, oracle.psi[i], oracle.w[i])
                gW, gb = oracle.g[i]
            ag.g_functions[i].weight.data.copy_(gW)
            ag.g_functions[i].bias.data.copy_(gb)
        hW, hb = (t(z['init.h.W']), t(z['init.h.b'])) if z is not None else oracle.h
        ag.h_function.weight.data.copy_(hW)
        ag.h_function.bias.data.copy_(hb)
    return dsf, ag


def cuda_tr(tr):
    return tuple(x.cuda() for x in tr)


def psi_params(sf, i, target=False):
    return [(lin.weight.data.cpu(), lin.bias.data.cpu()) for lin in linears(sf.psi[i][1 if target else 0][0].net)]


def gpi_rule(q, index):
    """
    The selection rule of the packed GPI keys (include/sfgpi.h, DESIGN.md "Packed keys") in float64: q [..., M] over M cells
    with index [M] -> the largest q, among the cells holding it the smallest index (-0 == +0); NaN is never selected; when
    every cell is NaN or -inf, index.min().  Returns (index [...], value [...]: the maximum, -inf in the last case).
    """
    v = torch.where(q.isnan(), torch.tensor(float('-inf'), dtype=q.dtype), q)
    m = v.max(dim=-1).values
    cand = (v == m.unsqueeze(-1)) & (m.unsqueeze(-1) > float('-inf'))
    pick = torch.where(cand, index, int(index.max()) + 1).min(dim=-1).values
    return torch.where(m == float('-inf'), index.min(), pick), m


def argmax_mismatch_ok(q_ref, idx_ref, idx_got, dim_pair, tol):
    """
    GPI argmax must be bit-exact except for ties inside tolerance: wherever the indices differ, the reference's top-1 and
    the value at our index must be within tol * max|q|.  q_ref [B,N,A]; dim_pair = 'task' | 'action'.
    """
    q_ref = q_ref.double()
    vals = q_ref.max(dim=2).values if dim_pair == 'task' else q_ref.max(dim=1).values       # [B,N] or [B,A]
    bad = (idx_ref.reshape(-1) != idx_got.reshape(-1)).nonzero().reshape(-1)
    scale = q_ref.abs().max()
    for b in bad.tolist():
        gap = vals[b, idx_ref.reshape(-1)[b]] - vals[b, idx_got.reshape(-1)[b]]
        if gap > tol * scale:
            return False, len(bad)
    return True, len(bad)
