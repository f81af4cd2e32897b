# -*- coding: UTF-8 -*-
"""
G1 "ensemble" generation of the reference (`source/features/deep.py` + `features/successor.py` + `agents/sfdqn.py:47-60`):
the only variant that trains ALL N psi networks on every replay batch -- the (transitions x tasks) unit of the headline
metric.  The reference loops `for index in range(n_tasks): sf.update_successor(transitions, index)` and re-runs GPI over all
N nets inside every iteration (N*(N+4) net passes); here `update_successors` does the whole thing in one fused pass
(5N net passes) with frozen-snapshot (Jacobi) semantics: every policy is stepped from the same pre-step library
(SURVEY.md section 3.4 / 8c; the literal Gauss-Seidel loop is still available through `update_successor(transitions, i)`).
"""
import torch

from .sfdqn import DeepSF as _DeepSF


class _RawW(torch.nn.Module):
    """Adapter so the packed reward row can be adopted like a Linear(D,1,bias=False)."""

    def __init__(self, w):
        super().__init__()
        self.weight = torch.nn.Parameter(w.reshape(1, -1).clone(), requires_grad=False)


class DeepSF(_DeepSF):
    """features/deep.py:8-131 on top of features/successor.py: raw-tensor w [D,1], LMS reward rule, l1-only psi update."""

    def __init__(self, pytorch_model_handle, *args, target_update_ev=1000, **kwargs):
        super().__init__(pytorch_model_handle, kwargs.pop('use_true_reward', False), target_update_ev, **kwargs)
        lr_sf = kwargs.get('learning_rate_sf', self.hyperparameters.get('learning_rate_sf', 1e-3))
        self.hyperparameters = dict(self.hyperparameters, learning_rate_sf=lr_sf)

    def add_training_task(self, task, source=None):
        true_w = torch.as_tensor(task.get_w()).float().to(self.device)
        n_features = task.feature_dim()
        if self.use_true_reward:
            fit_w = true_w.reshape(n_features, 1).clone()
        else:
            fit_w = torch.empty(n_features, 1, device=self.device).uniform_(-0.01, 0.01)     # features/successor.py:101
        holder = _RawW(fit_w)
        self.true_w.append(true_w)
        self.psi.append(self.build_successor(task, source, holder))
        self._w_holders = getattr(self, '_w_holders', []) + [holder]
        self.fit_w.append(holder.weight.data.view(n_features, 1))            # view of the packed row, shape [D,1]
        self.n_tasks = len(self.psi)
        import numpy as np
        for i in range(len(self.gpi_counters)):
            self.gpi_counters[i] = np.append(self.gpi_counters[i], 0)
        self.gpi_counters.append(np.zeros((self.n_tasks,), dtype=int))
        # growth may have re-packed the storage: refresh every raw view
        self.fit_w = [h.weight.data.view(-1, 1) for h in self._w_holders]

    def reset(self):
        super().reset()
        self._w_holders = []

    def load_state_dict(self, sd):
        super().load_state_dict(sd)
        self.fit_w = [h.weight.data.view(-1, 1) for h in self._w_holders]

    def update_reward(self, phi, r, task_index, exact=False):
        """LMS rule w += alpha_w (r - phi.w) phi, in place on the packed row (features/successor.py:146-167): one tiny kernel
        (sfgpi_lms_update) -- this is the per-environment-step op of main_sfdqn_torch.py."""
        import ctypes as C
        from . import _lib
        from .library import _stream
        w = self.fit_w[task_index]
        phi = torch.as_tensor(phi).float().to(self.device).reshape(-1).contiguous()
        r = torch.as_tensor(r).float().to(self.device).reshape(-1).contiguous()
        if phi.numel() != w.numel():
            raise ValueError('phi must have n_features elements')
        _lib.call('sfgpi_lms_update', w.data_ptr(), phi.data_ptr(), r.data_ptr(), w.numel(), float(self.alpha_w), _stream())
        if exact and not torch.allclose(r, torch.sum(phi.reshape(w.shape) * self.true_w[task_index].reshape(w.shape))):
            raise Exception('sampled reward {} != linear reward - please check task {}!'.format(r, task_index))

    def GPE_w(self, state, policy_index, w):
        return self.get_successor(state, policy_index) @ torch.as_tensor(w).float().to(self.device)

    def GPE(self, state, policy_index, task_index):
        return self.GPE_w(state, policy_index, self.fit_w[task_index])

    def update_successor(self, transitions, policy_index):
        """features/deep.py:93-131 for ONE policy (GPI over the whole library, l1 loss only)."""
        if transitions is None:
            return
        losses = self._library.train_step(transitions, policy_index, use_gpi=True, variant=0)
        self._after_update(policy_index)
        return losses[0, 0]

    def update_successors(self, transitions):
        """All N policies on one batch, one fused pass (the batched form of agents/sfdqn.py:59-60)."""
        if transitions is None:
            return
        losses = self._library.train_step(transitions, 'all', use_gpi=True, variant=0)
        for i in range(self.n_tasks):
            self._after_update(i)
        return losses[:, 0]
