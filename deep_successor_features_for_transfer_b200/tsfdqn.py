# -*- coding: UTF-8 -*-
"""
Drop-in for the reference's single-file G3 API (`source/tsfdqn.py`): ReplayBuffer, DeepTSF, TSFDQN (Transformed Successor
Features).  The TSF train step -- phi~ = phi * (h(g_i(s)) + h(g_i(s'))), target phi~ + gamma * psi^-(s', a*), loss
l1 + beta * l2, Adam over (psi_i, w_i, g_i, h) -- is one fused kernel sequence in libsfgpi.so (tsfdqn.py:588-709).
"""
import random

import numpy as np
import torch

import ctypes as C

from . import _lib
from .library import PackedSFLibrary, _stream
from .sfdqn import DeepSF, DeviceReplayBuffer, ReplayBuffer, SFDQN, _device  # noqa: F401  (re-exported like the reference file)


class PackedTargetOptim:
    """
    Adam over {w_target, omega} + the LambdaLR on omega's rate of one target task (tsfdqn.py:803-832) with all state on the
    device: moments, the step counter and the scheduler's epoch.  `step_fused` = update_test_reward_mapper + scheduler.step() as
    ONE kernel after the two ensemble forwards (csrc/target.cu: sfgpi_target_adapt).  `param_groups` / `scheduler` mimic what the
    agent's logging reads (tsfdqn.py:902-903).
    """

    class _Scheduler:
        def step(self):
            pass                                               # the epoch advances inside the fused kernel (tsfdqn.py:895)

    def __init__(self, w_approx, omegas, hp):
        dev = omegas.device
        self.hp = hp
        self.w_flat = w_approx.weight.data.reshape(-1).contiguous()
        w_approx.weight.data = self.w_flat.view(1, -1)
        z = lambda t: torch.zeros(t.numel(), dtype=torch.float32, device=dev)
        self.w_m, self.w_v, self.o_m, self.o_v = z(self.w_flat), z(self.w_flat), z(omegas), z(omegas)
        self.counters = torch.zeros(2, dtype=torch.int32, device=dev)              # [step, epoch]
        self.losses = torch.zeros(64, 3, dtype=torch.float32, device=dev)
        self.ring = 0
        self.scheduler = self._Scheduler()
        self._stage = torch.zeros(64, dtype=torch.float32, device=dev)

    @property
    def param_groups(self):
        epoch = int(self.counters[1])
        return [dict(lr=self.hp['learning_rate_w'], weight_decay=self.hp['weight_decay_w']),
                dict(lr=self.hp['learning_rate_omega'] * (1 - self.hp['learning_rate_omega_decay']) ** epoch,
                     weight_decay=self.hp['weight_decay_omega'])]

    def state_dict(self):
        """Adam state of (w, omega) -- clones of the moments, the shared step -- and the LambdaLR epoch.  The w and omega tensors
        themselves belong to the agent (TSFDQN.state_dict)."""
        step, epoch = (int(v) for v in self.counters.tolist())
        return dict(w_exp_avg=self.w_m.clone(), w_exp_avg_sq=self.w_v.clone(), omega_exp_avg=self.o_m.clone(),
                    omega_exp_avg_sq=self.o_v.clone(), step=step, last_epoch=epoch)

    def load_state_dict(self, sd):
        with torch.no_grad():
            for dst, k in ((self.w_m, 'w_exp_avg'), (self.w_v, 'w_exp_avg_sq'), (self.o_m, 'omega_exp_avg'), (self.o_v, 'omega_exp_avg_sq')):
                if tuple(sd[k].shape) != tuple(dst.shape):
                    raise ValueError(f"target-task optimizer state_dict: '{k}' has shape {tuple(sd[k].shape)}, expected {tuple(dst.shape)}")
                dst.copy_(sd[k])
            self.counters.copy_(torch.tensor([int(sd['step']), int(sd['last_epoch'])], dtype=torch.int32))

    def step_fused(self, agent, w_approx, omegas, phi, r, s, a, s1, a1):
        lib = agent.sf._library
        sp = lib.spec
        hp = self.hp
        if w_approx.weight.data.data_ptr() != self.w_flat.data_ptr() or not omegas.is_contiguous():
            raise ValueError('w_approx / omegas are not the tensors this optimizer was built for')
        with torch.no_grad():
            psi = lib.forward_psi(s, 0, lib.n)                                     # [1, N, A, D] online nets   (tsfdqn.py:948)
            next_psi = lib.forward_psi(s1, 0, lib.n, target=True)                  # target nets                (tsfdqn.py:950)
        if psi.shape[0] != 1:
            raise ValueError('the target-task step is a batch-1 update')
        t = _lib.TargetArgs()
        t.N, t.A, t.D, t.G, t.S = lib.n, sp.n_actions, sp.n_features, lib.G, sp.dims[0]
        t.psi, t.next_psi = psi.data_ptr(), next_psi.data_ptr()
        t.g, t.g_stride, t.h = lib.g.data_ptr(), lib.g.shape[1], lib.h.data_ptr()
        sv, s1v = s.reshape(-1).contiguous(), s1.reshape(-1).contiguous()
        phiv = phi.reshape(-1).contiguous()
        t.s, t.s1, t.phi = sv.data_ptr(), s1v.data_ptr(), phiv.data_ptr()
        t.r, t.gamma, t.a, t.a1 = float(r), float(agent.gamma), int(a), int(a1)
        t.beta, t.l1_coef = float(hp['beta_loss_coefficient']), float(hp['omegas_l1_coefficient'])
        t.lr_w, t.wd_w = float(hp['learning_rate_w']), float(hp['weight_decay_w'])
        t.lr_omega, t.wd_omega, t.lr_omega_decay = float(hp['learning_rate_omega']), float(hp['weight_decay_omega']), float(hp['learning_rate_omega_decay'])
        t.w, t.omegas = self.w_flat.data_ptr(), omegas.data_ptr()
        t.w_m, t.w_v, t.o_m, t.o_v = self.w_m.data_ptr(), self.w_v.data_ptr(), self.o_m.data_ptr(), self.o_v.data_ptr()
        t.step, t.epoch = self.counters.data_ptr(), self.counters.data_ptr() + 4
        self.ring = (self.ring + 1) % 64
        losses = self.losses[self.ring]
        t.losses = losses.data_ptr()
        _lib.call('sfgpi_target_adapt', C.byref(t), _stream())
        return losses[0], losses[1], losses[2]


class DeepTSF(DeepSF):
    """SF library of the TSF agent  [tsfdqn.py:93-324]: adds target-net forwards and the g/h optimizer groups."""

    def __init__(self, pytorch_model_handle, use_true_reward=False, target_update_ev=1000, **kwargs):
        super().__init__(pytorch_model_handle, use_true_reward, target_update_ev, **kwargs)
        self._tsf_dim = self.hyperparameters.get('g_h_function_dims')

    def add_training_task(self, task, source=None, g_function_model=None, h_function_model=None):
        if g_function_model is None or h_function_model is None:
            raise Exception('DeepTSF.add_training_task needs the g and h functions (tsfdqn.py:137)')
        if self._tsf_dim is None:
            self._tsf_dim = PackedSFLibrary._split_g(g_function_model)[1].out_features
            self._library = self._new_library()
        true_w = task.get_w()
        n_features = task.feature_dim()
        w_approx = torch.nn.Linear(n_features, 1, bias=False, device=self.device)
        with torch.no_grad():
            w_approx.weight.uniform_(-0.01, 0.01)
        self.true_w.append(true_w)
        self.fit_w.append(w_approx)
        self.psi.append(self.build_successor(task, source, w_approx, g_function_model, h_function_model))
        self.n_tasks = len(self.psi)
        for i in range(len(self.gpi_counters)):
            self.gpi_counters[i] = np.append(self.gpi_counters[i], 0)
        self.gpi_counters.append(np.zeros((self.n_tasks,), dtype=int))

    def get_next_successor(self, state, policy_index):
        return self._library.forward_psi(state, policy_index, 1, target=True)[:, 0]

    def get_next_successors(self, state):
        return self._library.forward_psi(state, 0, self.n_tasks, target=True)

    def update_successor(self, transitions, policy_index, use_gpi=True):
        raise Exception('This function should not be called')      # features/deep_sequential_tsf.py:184-185


class TSFDQN(SFDQN):
    """TSFDQN agent  [tsfdqn.py:329-1011]."""

    def __init__(self, deep_sf, buffer_handle, gamma, T, encoding, epsilon=0.1, epsilon_decay=1., epsilon_min=0.,
                 print_ev=1000, save_ev=100, use_gpi=True, test_epsilon=0.03, **kwargs):
        super().__init__(deep_sf, buffer_handle, gamma, T, encoding, epsilon, epsilon_decay, epsilon_min, print_ev, save_ev,
                         use_gpi, test_epsilon, **kwargs)
        self.omegas_per_source_task = []
        self.omegas = []
        self.g_functions = []
        self.h_function = None

    def reset(self):
        super().reset()
        self.g_functions = []
        self.h_function = None

    # ---- g / h / omega (tsfdqn.py:537-564) --------------------------------------------------------------------------
    def _init_g_function(self, states_dim, output_dim):
        return torch.nn.Linear(states_dim, output_dim, bias=True, device=self.device)

    def _init_h_function(self, input_dim, features_dim):
        return torch.nn.Linear(input_dim, features_dim, bias=True, device=self.device)

    def _init_omega(self, num_source_tasks):
        return torch.Tensor(1, num_source_tasks, 1, 1).uniform_(0, 1).to(self.device).requires_grad_(True)

    def add_training_task(self, task):
        self.tasks.append(task)
        self.n_tasks = len(self.tasks)
        self.phis.append(task.features)
        if self.n_tasks == 1:
            self.n_actions = task.action_count()
            self.n_features = task.feature_dim()
            if self.encoding == 'task':
                self.encoding = task.encode
        self.buffers.append(self.buffer_handle())
        g_h_function_dims = self.hyperparameters.get('g_h_function_dims')
        g_function = self._init_g_function(task.encode_dim(), g_h_function_dims)
        self.g_functions.append(g_function)
        if self.h_function is None:
            self.h_function = self._init_h_function(g_h_function_dims, task.feature_dim())
        self.sf.add_training_task(task, None, g_function, self.h_function)

    def set_active_training_task(self, index):
        super().set_active_training_task(index)
        self.active_g_function = self.g_functions[index]

    def get_Q_values(self, s, s_enc):
        with torch.no_grad():
            q, c = self.sf.GPI(s_enc, self.task_index, update_counters=self.use_gpi)
            if not self.use_gpi:
                c = self.task_index
            self.c = c
            return q[:, c, :]


    def _choose_action(self):
        """
        tsfdqn.py:453-457 + 416-432: unlike SFDQN.next_sample the TSF agent evaluates GPI on EVERY step (so gpi_counters move on
        exploratory steps too) and only then draws the epsilon-greedy coin.
        """
        greedy = self._greedy_action()
        if random.random() <= self.epsilon:
            a = torch.tensor(random.randrange(self.n_actions))
        else:
            a = greedy
        self.epsilon = max(self.epsilon * self.epsilon_decay, self.epsilon_min)
        return a

    # ---- the TSF train step -------------------------------------------------------------------------------------------
    def train_agent(self, s, s_enc, a, r, s1, s1_enc, gamma):
        phi = self.phi(s, a, s1)
        self.buffer.append(s_enc, a, r, phi, s1_enc, gamma)
        transitions = self.buffer.replay()
        losses = self.update_successor(transitions, self.task_index, self.use_gpi)
        if isinstance(losses, tuple) and self.logger is not None:
            total_loss, psi_loss, phi_loss = losses
            self.logger.log_losses(total_loss.item(), psi_loss.item(), phi_loss.item(),
                                   [self.hyperparameters['beta_loss_coefficient']], self.total_training_steps)

    def update_successor(self, transitions, policy_index, use_gpi=True):
        if transitions is None:
            return
        if self.h_function is None:
            raise Exception('Affine Function (h) is not initialized')
        beta = self.hyperparameters['beta_loss_coefficient']
        losses = self.sf._library.train_step(transitions, policy_index, use_gpi=use_gpi, variant=2, beta=beta)
        self.sf._after_update(policy_index)
        return losses[0, 0], losses[0, 1], losses[0, 2]

    def update_successor_all(self, transitions, use_gpi=True, host_losses=None):
        """
        Ensemble extension (BASELINE config 4-ii): all policies stepped on one batch, frozen-snapshot semantics.  Returns the
        losses [n_tasks][3] on the device; with host_losses (a pinned CPU float32 tensor of that shape) the step also copies
        them there asynchronously -- synchronise the current stream before reading it.
        """
        if transitions is None:
            return
        beta = self.hyperparameters['beta_loss_coefficient']
        losses = self.sf._library.train_step(transitions, 'all', use_gpi=use_gpi, variant=2, beta=beta, host_losses=host_losses)
        for i in range(self.sf.n_tasks):
            self.sf._after_update(i)
        return losses

    # ---- target tasks: omega-weighted transfer (tsfdqn.py:784-1011; SURVEY 8f N1) -----------------------------------------
    # Host loop as in the reference; every psi evaluation (get_successors / get_next_successors: N nets per call) runs on the
    # fused ensemble kernels, the (w, omega) update is a handful of [1, N, A, D]-sized torch ops.
    def _epsilon_greedy(self, q):
        q = q.flatten()
        assert q.size()[0] == self.n_actions
        if random.random() <= self.epsilon:
            a = torch.tensor(random.randrange(self.n_actions)).to(self.device)
        else:
            a = torch.argmax(q)
        self.epsilon = max(self.epsilon * self.epsilon_decay, self.epsilon_min)
        return a

    def _new_target_task(self, feature_dim, omegas_init, fused=True):
        """
        (w_approx, Adam over {w, omega}, LambdaLR decaying only omega's lr, omegas) for one target task (tsfdqn.py:803-832).
        fused (default): the optimizer / scheduler are views of a PackedTargetOptim -- moments, step and the scheduler's epoch live
        on the device and update_test_reward_mapper runs as ONE kernel (csrc/target.cu); fused=False builds the reference's own
        torch.optim.Adam + LambdaLR (the eager path, kept for callers that hand in their own optimizer).
        """
        hp = self.hyperparameters
        if fused and self.sf._library.n_flows > 0:
            fused = False                                     # the fused target kernel evaluates a LINEAR g (csrc/target.cu)
        if fused:
            omegas = omegas_init.clone().detach().to(self.device).float().contiguous()
            w_approx = torch.nn.Linear(feature_dim, 1, bias=False, device=self.device)
            with torch.no_grad():
                w_approx.weight.uniform_(-0.01, 0.01)
            optim = PackedTargetOptim(w_approx, omegas, hp)
            return w_approx, optim, optim.scheduler, omegas
        omegas = omegas_init.clone().detach().requires_grad_(True)
        w_approx = torch.nn.Linear(feature_dim, 1, bias=False, device=self.device)
        with torch.no_grad():
            w_approx.weight.uniform_(-0.01, 0.01)
        optim = torch.optim.Adam([
            {'params': w_approx.parameters(), 'lr': hp['learning_rate_w'], 'weight_decay': hp['weight_decay_w']},
            {'params': omegas, 'lr': hp['learning_rate_omega'], 'weight_decay': hp['weight_decay_omega']}])
        decay = hp['learning_rate_omega_decay']
        scheduler = torch.optim.lr_scheduler.LambdaLR(optim, [lambda epoch: 1.0, lambda epoch: (1 - decay) ** epoch])
        return w_approx, optim, scheduler, omegas

    def _test_task_state(self, k):
        """Target task k: w, omega and their optimizer (a PackedTargetOptim, or torch.optim.Adam + LambdaLR)."""
        w, optim, scheduler = self.test_tasks_weights[k]
        fused = isinstance(optim, PackedTargetOptim)
        return dict(w=w.weight.detach().clone(), omegas=self.omegas[k].detach().clone(), fused=fused, optim=optim.state_dict(),
                    scheduler=None if fused else scheduler.state_dict())

    def _load_test_task(self, k, tsd):
        if k == len(self.test_tasks_weights):
            w, optim, scheduler, omegas = self._new_target_task(tsd['w'].numel(), tsd['omegas'].to(self.device), fused=tsd['fused'])
            self.test_tasks_weights.append((w, optim, scheduler))
            self.omegas.append(omegas)
        w, optim, scheduler = self.test_tasks_weights[k]
        if isinstance(optim, PackedTargetOptim) != tsd['fused']:
            raise ValueError(f'agent state_dict: target task {k} was saved with a '
                             f"{'fused' if tsd['fused'] else 'torch.optim.Adam'} optimizer, this agent has the other kind")
        with torch.no_grad():
            w.weight.copy_(tsd['w'].reshape(w.weight.shape))
            self.omegas[k].copy_(tsd['omegas'])
        optim.load_state_dict(tsd['optim'])
        if tsd['scheduler'] is not None:
            scheduler.load_state_dict(tsd['scheduler'])

    def train(self, train_tasks, n_samples, viewers=None, n_view_ev=None, test_tasks=[], n_test_ev=1000, cycles_per_task=1):
        if viewers is None:
            viewers = [None] * len(train_tasks)
        self.reset()
        for train_task in train_tasks:
            self.add_training_task(train_task)
        with torch.no_grad():
            omegas0 = self._init_omega(len(train_tasks))
            omegas0 = omegas0 / torch.sum(omegas0, axis=1, keepdim=True)          # sum_i omega_i = 1 at the start
        self.test_tasks_weights, self.omegas = [], []
        for test_task in test_tasks:
            w_approx, optim, scheduler, omegas = self._new_target_task(test_task.feature_dim(), omegas0)
            self.test_tasks_weights.append((w_approx, optim, scheduler))
            self.omegas.append(omegas)
        return_data = []
        for _ in range(cycles_per_task):
            for index, (train_task, viewer) in enumerate(zip(train_tasks, viewers)):
                self.set_active_training_task(index)
                for t in range(n_samples):
                    self.next_sample(viewer, n_view_ev)
                    if t % n_test_ev == 0 and len(test_tasks) > 0:
                        Rs = [self.test_agent(task, k) for k, task in enumerate(test_tasks)]
                        avg_R = torch.mean(torch.Tensor(Rs).to(self.device))
                        return_data.append(avg_R)
                        if self.logger is not None:
                            self.logger.log_progress(self.get_progress_dict())
                            self.logger.log_average_reward(avg_R, self.total_training_steps)
                            self.logger.log_accumulative_reward(torch.sum(torch.Tensor(return_data).to(self.device)),
                                                                self.total_training_steps)
                    self.total_training_steps += 1
        return return_data

    @staticmethod
    def _normalized(omegas):
        return omegas / torch.sum(omegas, axis=1, keepdim=True)

    def get_test_action(self, s_enc, w, omegas=None):
        if omegas is None:                                    # SFDQN-style call (GPI over the library under w)
            return super().get_test_action(s_enc, w)
        with torch.no_grad():
            if random.random() <= self.test_epsilon:
                return torch.tensor(random.randrange(self.n_actions)).to(self.device)
            lib = self.sf._library
            psi = self.sf.get_successors(s_enc)                                   # [1, N, A, D]  (ensemble kernel)
            if psi.shape[0] != 1:
                tsf = torch.sum(psi * self._normalized(omegas), axis=1)
                return torch.argmax(w(tsf))
            # fused: q = w(sum_j omega^_j psi_j(s)) and its argmax in one kernel (csrc/target.cu)
            act = lib._ws.get('target_action')
            if act is None:
                act = lib._ws['target_action'] = torch.empty(1, dtype=torch.int64, device=self.device)
            wv = w.weight if isinstance(w, torch.nn.Module) else w
            _lib.call('sfgpi_target_q', psi.data_ptr(), psi.shape[1], psi.shape[2], psi.shape[3],
                      omegas.detach().contiguous().data_ptr(), wv.detach().contiguous().data_ptr(), None, act.data_ptr(), _stream())
            return act[0].clone()                             # the target task acts by Q-learning on the mixed psi

    def test_agent(self, task, test_index):
        R = 0.0
        w, optim, scheduler = self.test_tasks_weights[test_index]
        omegas = self.omegas[test_index]
        s_enc = self.encoding(task.initialize())
        accum = [0.0, 0.0, 0.0]
        for _ in range(self.T):
            a = self.get_test_action(s_enc, w, omegas)
            s1, r, done = task.transition(a)
            s1_enc = self.encoding(s1)
            a1 = self.get_test_action(s1_enc, w, omegas)
            losses = self.update_test_reward_mapper(w, omegas, optim, task, r, s_enc, a, s1_enc, a1)
            accum = [acc + float(x) for acc, x in zip(accum, losses)]
            scheduler.step()
            s_enc = s1_enc
            R += r
            if done:
                break
        if self.total_training_steps % 5000 == 0 and self.logger is not None:
            beta = self.hyperparameters['beta_loss_coefficient']
            self.logger.log_target_error_progress(
                self.get_target_reward_mapper_error(R, accum[0], accum[1], accum[2], test_index, beta, self.T))
            self.logger.log_omegas_learning_rate(optim.param_groups[1]['lr'], test_index, self.total_training_steps)
        self.omegas[test_index] = omegas
        return R

    def update_test_reward_mapper(self, w_approx, omegas, optim, task, r, s, a, s1, a1=None):
        """One (w, omega) step on a target task: returns (loss, reward loss, psi loss)  [tsfdqn.py:917-997]."""
        if self.h_function is None:
            raise Exception('Affine Function (h) is not initialized')
        hp = self.hyperparameters
        s, s1 = torch.as_tensor(s).float().to(self.device), torch.as_tensor(s1).float().to(self.device)
        phi = torch.as_tensor(task.features(s, a, s1)).float().to(self.device)
        if isinstance(optim, PackedTargetOptim):
            return optim.step_fused(self, w_approx, omegas, phi, r, s, a, s1, a1)
        norm = self._normalized(omegas)
        with torch.no_grad():
            ts = torch.vstack([g(s) for g in self.g_functions]).unsqueeze(1)          # [N, 1, G] -> broadcasts with [1, N, 1, 1]
            ts1 = torch.vstack([g(s1) for g in self.g_functions]).unsqueeze(1)
            psi = self.sf.get_successors(s)                                           # [1, N, A, D]  (ensemble kernel)
            next_psi = self.sf.get_next_successors(s1)                                # target nets
            r_tensor = torch.tensor(r).float().unsqueeze(0).to(self.device)
        affine = self.h_function(torch.sum(ts * norm, axis=1)) + self.h_function(torch.sum(ts1 * norm, axis=1))
        tphi = phi * affine.squeeze(0)
        next_tsf = tphi + self.gamma * torch.sum(next_psi * norm, axis=1)[:, a1, :]
        tsf = torch.sum(psi * norm, axis=1)[:, a, :]
        l1 = torch.nn.functional.mse_loss(tsf, next_tsf)
        l2 = torch.mean((w_approx(tphi) - r_tensor) ** 2)
        loss = l1 + hp['beta_loss_coefficient'] * l2 + hp['omegas_l1_coefficient'] * torch.norm(omegas, 1)
        optim.zero_grad()
        loss.backward()
        optim.step()
        with torch.no_grad():
            omegas.clamp_(1e-7)
        return loss, l2, l1

    def get_target_reward_mapper_error(self, r, loss, phi_loss, psi_loss, task_index, target_loss_coefficient, ts):
        return {'task': task_index, 'reward': r, 'steps': (500 * (self.total_training_steps // 1000)) + ts, 'w_error': loss,
                'psi_loss': psi_loss, 'phi_loss': phi_loss, 'target_loss_coefficient': target_loss_coefficient}

    def get_progress_strings(self):
        sample_str = 'task \t {} \t steps \t {} \t episodes \t {} \t eps \t {:.4f}'.format(
            self.task_index, self.steps, self.episode, self.epsilon)
        reward_str = 'ep_reward \t {:.4f} \t reward \t {:.4f}'.format(self.episode_reward, self.reward)
        w_error = torch.linalg.norm(self.sf.fit_w[self.task_index].weight.T -
                                    torch.as_tensor(self.sf.true_w[self.task_index]).to(self.device))
        gpi_str = 'GPI% \t {:.4f} \t w_err \t {:.4f}'.format(self.sf.GPI_usage_percent(self.task_index), w_error)
        return sample_str, reward_str, gpi_str
