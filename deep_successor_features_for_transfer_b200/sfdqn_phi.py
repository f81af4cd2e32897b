# -*- coding: UTF-8 -*-
"""
Learned features (phi): drop-in for the reference's `PhiFunction` and `SFDQN.pre_train` (source/sfdqn_phi.py:90-123, 800-873;
SURVEY 8f N3).  phi_theta(cat[s, a, s']) is a small MLP (2S + action_dim -> 128 -> 256 -> D, ReLU) regressed so that the
per-task linear heads w_i reproduce the rewards: loss = mse_loss(r, w_i(phi_theta(s, a, s'))), one Adam for theta (stepped at
every update) and one Adam per head (stepped when its task's batch is used).

Here one update is a replayed command list of libsfgpi.so -- fused MLP forward (sfgpi_mlp_forward, activations saved), the
regression head (sfgpi_phi_head: loss partials, dL/dphi, dL/dw), the MLP backward (sfgpi_mlp_backward), and two Adam steps
(sfgpi_adam_step; the head's also reduces the loss) -- on the parameters packed in a one-row `PackedSFLibrary` (fp32 mode:
the layer widths are not the 256-wide tensor-core shape, and at B = 32 the step is launch-latency-bound anyway).
The replay ring, the random-policy rollout and the task protocol stay host-side Python, as in the reference.
"""
import ctypes as C
import math
import random

import torch

from . import _lib
from .library import PackedSFLibrary, _stream
from .sfdqn import DeepSF, ReplayBuffer, _device


class _RewardHead:
    """fit_w = Linear(D, 1, bias=False) with U(-0.01, 0.01) weights + its own Adam(lr=1e-3)  (sfdqn_phi.py:819-826)."""

    def __init__(self, feature_dim, device, lr=1e-3):
        lin = torch.nn.Linear(feature_dim, 1, bias=False)                       # consumes the RNG like the reference's does
        with torch.no_grad():
            lin.weight = torch.nn.Parameter(torch.Tensor(1, feature_dim).uniform_(-0.01, 0.01))
        self.module = lin
        self.lr = lr
        self.weight = lin.weight.data.reshape(-1).to(device).contiguous()       # [D] on the device; the module views it
        lin.weight.data = self.weight.view(1, -1)
        self.m, self.v = torch.zeros_like(self.weight), torch.zeros_like(self.weight)
        self.step = torch.zeros(1, dtype=torch.int32, device=device)
        self.consts = torch.tensor([[1.0 - 0.9 ** 1, math.sqrt(1.0 - 0.999 ** 1)]], dtype=torch.float64, device=device)


class PhiFunction:
    """
    phi_theta(state, action, next_state) -> [B, feature_dimension]  (sfdqn_phi.py:90-123).  Same constructor arguments,
    `forward` / call semantics (0-/1-dim actions and 1-dim states are promoted like the reference does), `set_eval()`,
    `alpha_phi`, and `_model` (an nn.Sequential whose parameters are views of the packed row, so `.parameters()` /
    `state_dict()` keep working).
    """

    def __init__(self, state_space, action_space, feature_dimension):
        self.alpha_phi = 1e-3
        self.device = _device()
        self.in_dim, self.D = state_space * 2 + action_space, feature_dimension
        layers = [torch.nn.Linear(self.in_dim, 128), torch.nn.ReLU(), torch.nn.Linear(128, 128 * 2), torch.nn.ReLU(),
                  torch.nn.Linear(128 * 2, feature_dimension)]
        self._model = torch.nn.Sequential(*layers)
        rng = torch.get_rng_state()                                              # (the storage twin must not advance the RNG)
        twin = torch.nn.Sequential(*[torch.nn.Linear(l.in_features, l.out_features) if isinstance(l, torch.nn.Linear)
                                     else torch.nn.ReLU() for l in layers])
        self._library = PackedSFLibrary(device=self.device, lr=dict(sf=self.alpha_phi, w=1e-3, g=1e-3, h=1e-3), capacity=1,
                                        precision='fp32')
        w_stub = torch.nn.Linear(feature_dimension, 1, bias=False)
        torch.set_rng_state(rng)
        twin.load_state_dict(self._model.state_dict())
        self._library.add_policy(self._model, twin, w_stub, n_actions=1, n_features=feature_dimension)
        self._library._point_views(0, self._library._views[0])
        self._model.train()
        self._plans = {}

    # ---- forward ----------------------------------------------------------------------------------------------------
    def _inputs(self, state, action, next_state):
        dev = self.device
        state, next_state = torch.as_tensor(state).to(dev), torch.as_tensor(next_state).to(dev)
        action = torch.as_tensor(action).to(dev)
        if action.ndim == 0:
            action = action.unsqueeze(0)
        if action.ndim == 1:
            action = action.unsqueeze(1)
        if state.ndim == 1:
            state = state.unsqueeze(0)
        if next_state.ndim == 1:
            next_state = next_state.unsqueeze(0)
        return torch.cat([state, action, next_state], axis=1).float().contiguous()     # sfdqn_phi.py:116

    def forward(self, state, action, next_state):
        x = self._inputs(state, action, next_state)
        return self._library.forward_psi(x, 0, 1).reshape(x.shape[0], self.D)

    __call__ = forward

    def set_eval(self):
        self._model.eval()

    # ---- one regression update (the body of pre_train's inner loop, sfdqn_phi.py:848-866) ------------------------------
    def _plan(self, B):
        plan = self._plans.get(B)
        if plan is not None:
            return plan
        lib, sp, dev = self._library, self._library.spec, self.device
        D = self.D
        ws = lib._workspace(B, 1)
        nblk = _lib.lib().sfgpi_phi_head_partials(B)
        f = lambda *shape: torch.zeros(*shape, dtype=torch.float32, device=dev)
        buf = dict(x=f(B, self.in_dim), r=f(B), phi=f(B, D), d_out=f(1, B, D), dw=f(nblk, D), lp=f(nblk, 2),
                   zeros=torch.zeros(B, dtype=torch.int64, device=dev), losses=f(64, 1, 3), ring=0)
        a = lib._fwd_args(lib.online, 0, 1, buf['x'])
        a.psi_out = buf['phi'].data_ptr()
        lib._save_acts(a, ws['acts'], ws['masks'])
        b, _, _ = lib._backward_args(ws, 0, 1, B)
        b.x, b.actions, b.d_out = buf['x'].data_ptr(), buf['zeros'].data_ptr(), buf['d_out'].data_ptr()

        def adam(param, m, v, length, grad, n_part, part_stride, lr, step, consts):
            ad = _lib.AdamArgs()
            ad.n_seg, ad.n_pol, ad.step, ad.consts = 1, 1, step.data_ptr(), consts.data_ptr()
            ad.beta1, ad.beta2, ad.eps = 0.9, 0.999, 1e-8
            s = ad.seg[0]
            s.param, s.m, s.v, s.param_stride, s.m_stride, s.v_stride = param, m, v, length, length, length
            s.grad_part, s.grad_pol_stride, s.grad_part_stride, s.n_part = grad, n_part * part_stride, part_stride, n_part
            s.len, s.lr, s.weight_decay = length, lr, 0.0
            ad.sequential_shared = 1
            return ad

        rs = sp.row_stride
        ad_phi = adam(lib.online.data_ptr(), lib.m.data_ptr(), lib.v.data_ptr(), rs, ws['grad_part'].data_ptr(), ws['n_split'], rs,
                      self.alpha_phi, lib.step, lib.adam_consts)
        plan = self._plans[B] = dict(buf=buf, a=a, b=b, ad_phi=ad_phi, nblk=nblk, B=B, ws=ws, adam=adam)
        return plan

    def regression_step(self, state, action, reward, next_state, head, loss_slot=None):
        """
        phis = phi(s, a, s'); loss = mse_loss(reward, head(phis)); backward; phi's Adam and the head's Adam step.
        Returns the loss as a 0-dim device tensor (no host sync): a view of `loss_slot` ([1, 3] fp32, device) when given, else
        of one slot of a 64-deep ring (valid for the next 63 updates).
        """
        x = self._inputs(state, action, next_state)
        B = x.shape[0]
        reward = torch.as_tensor(reward).to(self.device).float().reshape(-1)
        if reward.numel() != B:
            raise ValueError('one reward per transition expected')
        plan = self._plan(B)
        buf, st = plan['buf'], _stream()
        buf['x'].copy_(x)
        buf['r'].copy_(reward)
        D = self.D
        _lib.call('sfgpi_mlp_forward', C.byref(plan['a']), st)
        _lib.call('sfgpi_phi_head', buf['phi'].data_ptr(), head.weight.data_ptr(), buf['r'].data_ptr(), B, D, buf['d_out'].data_ptr(),
                  buf['dw'].data_ptr(), buf['lp'].data_ptr(), st)
        _lib.call('sfgpi_mlp_backward', C.byref(plan['b']), st)
        _lib.call('sfgpi_adam_step', C.byref(plan['ad_phi']), st)
        if loss_slot is None:
            buf['ring'] = (buf['ring'] + 1) % 64
            losses = buf['losses'][buf['ring']]
        else:
            losses = loss_slot
        ad_w = plan['adam'](head.weight.data_ptr(), head.m.data_ptr(), head.v.data_ptr(), D, buf['dw'].data_ptr(), plan['nblk'], D,
                            head.lr, head.step, head.consts)
        ad_w.loss_part, ad_w.n_loss_part = buf['lp'].data_ptr(), plan['nblk']
        ad_w.l1_scale, ad_w.l2_scale, ad_w.beta_loss, ad_w.losses = 0.0, 1.0 / B, 1.0, losses.data_ptr()
        _lib.call('sfgpi_adam_step', C.byref(ad_w), st)
        return losses[0, 0]


def pre_train(train_tasks, n_samples_pre_train, n_cycles=5, buffer_handle=None):
    """
    SFDQN.pre_train (sfdqn_phi.py:800-873): fits phi on random-policy rollouts of the training tasks.  Returns
    (phi_learn_model, losses) -- the reference stores the model in `self.learnt_phi` and returns the losses; the host loop,
    the RNG consumption order (torch for the initialisations, `random` for the actions, numpy for the replay picks) and the
    replay ring are the reference's.
    """
    device = _device()
    first_task = train_tasks[0]
    buffer = ReplayBuffer() if buffer_handle is None else buffer_handle()
    n_actions = first_task.action_count()
    phi_learn_model = PhiFunction(first_task.encode_dim(), first_task.action_dim(), first_task.feature_dim())
    heads = [_RewardHead(task.feature_dim(), device) for task in train_tasks]
    losses = []
    log = torch.zeros(max(1, n_cycles * len(train_tasks) * n_samples_pre_train), 1, 3, dtype=torch.float32, device=device)
    for cycle in range(n_cycles):
        for task_id, task in enumerate(train_tasks):
            head = heads[task_id]
            s_enc = task.encode(task.initialize())
            for sample in range(n_samples_pre_train):
                a = random.randrange(n_actions)
                s1, r, terminal = task.transition(a)
                s1_enc = task.encode(s1)
                buffer.append(s_enc, torch.tensor(a), torch.tensor(r, dtype=torch.float32), torch.tensor([0]), s1_enc, torch.tensor([0]))
                s_enc = s1_enc
                if terminal:
                    s_enc = task.encode(task.initialize())
                replay = buffer.replay()
                if replay is not None:
                    state_batch, action_batch, reward_batch, _, next_state_batch, _ = replay
                    losses.append(phi_learn_model.regression_step(state_batch, action_batch, reward_batch, next_state_batch, head,
                                                                  loss_slot=log[len(losses)]))
    buffer.reset()
    phi_learn_model.set_eval()
    phi_learn_model.reward_heads = heads
    return phi_learn_model, [float(v) for v in log[:len(losses), 0, 0].cpu()]      # (the reference syncs on loss.item() per update)


class PackedPhi(torch.nn.Module):
    """
    A phi network (any Linear / ReLU / Tanh nn.Sequential, e.g. main_sfdqn_phi_torch.py:52-73's 5-layer MLP over cat[s, a, s'])
    adopted into a one-row packed library so that the G4 / G5 joint step can run it on the kernels.  Parameters are views of the
    packed row (`.parameters()`, `state_dict()` keep working); calling it runs the fused CUDA forward.
    """

    def __init__(self, model, feature_dim):
        super().__init__()
        self.net = model
        dev = _device()
        rng = torch.get_rng_state()
        twin = torch.nn.Sequential(*[torch.nn.Linear(l.in_features, l.out_features) if isinstance(l, torch.nn.Linear) else type(l)()
                                     for l in model.children()])
        lib = PackedSFLibrary(device=dev, capacity=1, precision='fp32')
        w_stub = torch.nn.Linear(feature_dim, 1, bias=False)
        torch.set_rng_state(rng)
        twin.load_state_dict(model.state_dict())
        lib.add_policy(model, twin, w_stub, n_actions=1, n_features=feature_dim)
        lib._point_views(0, lib._views[0])
        self._lib_ref = [lib]
        self.feature_dim = feature_dim

    @property
    def library(self):
        return self._lib_ref[0]

    def forward(self, x):
        x = torch.as_tensor(x).to(_device()).float().contiguous()
        return self.library.forward_psi(x, 0, 1).reshape(x.shape[0], self.feature_dim)


class DeepSF_PHI(DeepSF):
    """
    SF library of the phi-learning agents, G4 (features/deep_phi.py:11-290): fit_w[i] = Linear(D, 1) WITH bias
    (:266-270), GPI's q = w(psi)[..., 0] includes that bias (:248), and update_successor is the JOINT psi / phi step
    (:95-224) -- here one kernel sequence (PackedSFLibrary.train_step_g4) instead of ~100 eager ops and a freshly built
    torch.optim.Adam per call.
    """

    _eager_step_unsupported = 'DeepSF_PHI (its step is the joint psi / phi update)'

    def add_training_task(self, task, source=None):
        n_features = task.feature_dim()
        self.psi.append(None)                                                     # (reference order: psi nets first, then fit_w, :262-270)
        w_holder = torch.nn.Linear(n_features, 1, bias=False, device=self.device)
        self.psi[-1] = self.build_successor(task, source, w_holder)
        self.n_tasks = len(self.psi)
        fit_w = torch.nn.Linear(n_features, 1).to(self.device)
        with torch.no_grad():
            self._library.w[self.n_tasks - 1].copy_(fit_w.weight.data.reshape(-1))
        fit_w.weight.data = self._library.w[self.n_tasks - 1].view(1, -1)          # view of the packed row
        self._library._views[self.n_tasks - 1]['w'] = fit_w
        self.fit_w.append(fit_w)
        self.true_w.append(task.get_w())
        import numpy as np
        for i in range(len(self.gpi_counters)):
            self.gpi_counters[i] = np.append(self.gpi_counters[i], 0)
        self.gpi_counters.append(np.zeros((self.n_tasks,), dtype=int))

    def GPI_w(self, state, w):
        q, task = super().GPI_w(state, w)
        if isinstance(w, torch.nn.Module) and getattr(w, 'bias', None) is not None:
            q = q + w.bias.detach().to(q.device)                                   # w(psi): the bias shifts every cell equally
        return q, task

    def update_reward(self, phi, r, task_index, exact=False):
        raise Exception('This function should not be used')                        # features/deep_phi.py:92-93

    def update_successor(self, transitions, phis_model, policy_index, loss_coefficient, use_gpi=True):
        if transitions is None:
            return
        (phi_model, _, _), _ = phis_model
        if not isinstance(phi_model, PackedPhi):
            raise TypeError('the phi model must be a PackedPhi (wrap the nn.Sequential the phi lambda returns)')
        fit_w = self.fit_w[policy_index]
        losses = self._library.train_step_g4(transitions, policy_index, phi_model.library, fit_w.bias.data, loss_coefficient.data,
                                             use_gpi=use_gpi)
        self._after_update(policy_index)
        return losses[0:1], losses[1:2], losses[2:3], loss_coefficient
