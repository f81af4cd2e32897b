# -*- coding: UTF-8 -*-
"""
Drop-in for the reference's single-file G2 API (`source/sfdqn.py`): ReplayBuffer, DeepSF, SFDQN -- same constructor
arguments, method names, return shapes and error behaviour -- with the hot path (psi forward over the policy ensemble, GPI,
TD target, backward, Adam) executed by hand-written sm_100a kernels through libsfgpi.so instead of eager PyTorch.

What stays host-side Python (as in the reference): the replay ring, epsilon-greedy, environment stepping, logging.
"""
import random
from collections import OrderedDict

import numpy as np
import torch

from .library import ADAM_BETA1, ADAM_BETA2, ADAM_EPS, PackedSFLibrary


def _device():
    if not torch.cuda.is_available():
        raise RuntimeError('no CUDA device: the B200 SF/GPI path has no CPU fallback')
    return torch.device('cuda', torch.cuda.current_device())


class ReplayBuffer:
    """Randomised replay ring with the reference's tuple order (s, a, r, phi, s', gamma)  [sfdqn.py:12-89]."""

    def __init__(self, n_samples=1000000, n_batch=32):
        self.n_samples = n_samples
        self.n_batch = n_batch
        self.reset()

    def reset(self):
        self.buffer = np.empty(self.n_samples, dtype=object)
        self.index = 0
        self.size = 0

    def replay(self):
        """None until n_batch samples exist (sfdqn.py:57); else (states, actions, rewards, phis, next_states, gammas)."""
        if self.size < self.n_batch:
            return None
        picks = np.random.randint(low=0, high=self.size, size=(self.n_batch,))
        cols = list(zip(*self.buffer[picks]))
        dev = _device()
        stack = lambda c: torch.vstack([torch.as_tensor(v) for v in c]).to(dev)
        flat = lambda c: torch.as_tensor(np.asarray([float(v) if not torch.is_tensor(v) else v.item() for v in c]))
        states, rewards, phis, next_states = stack(cols[0]), stack(cols[2]), stack(cols[3]), stack(cols[4])
        actions = torch.as_tensor(np.asarray([int(v) for v in cols[1]], dtype=np.int64)).to(dev)
        gammas = flat(cols[5]).float().to(dev)
        return states, actions, rewards, phis, next_states, gammas

    def append(self, state, action, reward, phi, next_state, gamma):
        reward = torch.as_tensor(reward).float()          # rewards arrive as doubles (sfdqn.py:86)
        self.buffer[self.index] = (state, action, reward, phi, next_state, gamma)
        self.size = min(self.size + 1, self.n_samples)
        self.index = (self.index + 1) % self.n_samples

    def state_dict(self):
        """Slots [:size] as stacked tensors (states / next_states [size][S], actions int64, rewards / gammas [size], phis
        [size][D]) with the write index and the size: the format DeviceReplayBuffer uses too, so either ring loads the other's."""
        cols = list(zip(*self.buffer[:self.size])) if self.size else [()] * 6
        stack = lambda c: torch.vstack([torch.as_tensor(v) for v in c]) if c else torch.empty(0)
        return dict(n_samples=self.n_samples, index=self.index, size=self.size, states=stack(cols[0]),
                    actions=torch.as_tensor([int(v) for v in cols[1]], dtype=torch.int64), rewards=stack(cols[2]).reshape(-1),
                    phis=stack(cols[3]), next_states=stack(cols[4]),
                    gammas=torch.as_tensor([float(v) for v in cols[5]], dtype=torch.float64))

    def load_state_dict(self, sd):
        _check_ring_dict(self, sd)
        self.reset()
        cpu = {k: sd[k].detach().cpu() for k in _RING_FIELDS}
        for k in range(sd['size']):
            self.buffer[k] = (cpu['states'][k:k + 1], int(cpu['actions'][k]), cpu['rewards'][k].float(), cpu['phis'][k],
                              cpu['next_states'][k:k + 1], float(cpu['gammas'][k]))
        self.index, self.size = int(sd['index']), int(sd['size'])


_RING_FIELDS = ('states', 'actions', 'rewards', 'phis', 'next_states', 'gammas')


def _check_ring_dict(ring, sd):
    for k in ('n_samples', 'index', 'size') + _RING_FIELDS:
        if k not in sd:
            raise ValueError(f"replay state_dict: missing key '{k}'")
    if int(sd['n_samples']) != ring.n_samples:
        raise ValueError(f"replay state_dict: saved from a ring of {sd['n_samples']} samples, this ring holds {ring.n_samples}")
    if any(sd[k].shape[0] != sd['size'] for k in _RING_FIELDS) or not 0 <= sd['index'] < ring.n_samples:
        raise ValueError('replay state_dict: inconsistent sizes')


class DeviceReplayBuffer:
    """
    Same interface and sampling stream as ReplayBuffer (sfdqn.py:12-89), but the ring lives in HBM as packed fp32 rows
    [s | s' | phi | r | gamma | action] and replay() is ONE gather kernel (csrc/replay.cu) instead of python loops + vstack +
    .to(device) (66 ms per B=4096 batch in the reference, SURVEY 8f N2).  Picks come from np.random.randint exactly like the
    reference's, so under the same numpy seed both buffers return the same transitions.
    """

    def __init__(self, n_samples=1000000, n_batch=32):
        self.n_samples = int(n_samples)
        self.n_batch = int(n_batch)
        self.reset()

    def reset(self):
        self.ring = None
        self.index = 0
        self.size = 0
        self._out = None

    def _alloc(self, S, D):
        import ctypes as C
        from . import _lib
        dev = _device()
        self.S, self.D = S, D
        self.row = 2 * S + D + 3
        self.ring = torch.zeros(self.n_samples, self.row, dtype=torch.float32, device=dev)
        B = self.n_batch
        f32 = lambda *shape: torch.empty(*shape, dtype=torch.float32, device=dev)
        self._out = (f32(B, S), torch.empty(B, dtype=torch.int64, device=dev), f32(B, 1), f32(B, D), f32(B, S), f32(B))
        self._picks = torch.empty(B, dtype=torch.int64, device=dev)
        # pinned staging of the picks: a small ring, each slot guarded by the event of the copy that last read it, so a host
        # that runs ahead of the stream (replay -> train_step loops never synchronise) cannot rewrite picks still in flight
        self._picks_host = [torch.empty(B, dtype=torch.int64).pin_memory() for _ in range(4)]
        self._picks_done = [None] * 4
        self._picks_slot = 0
        self._row_host = [torch.empty(self.row, dtype=torch.float32).pin_memory() for _ in range(16)]
        self._row_done = [None] * 16
        self._row_slot = 0
        a = self._args = _lib.ReplayArgs()
        a.ring, a.row_stride, a.S, a.D, a.B, a.picks = self.ring.data_ptr(), self.row, S, D, B, self._picks.data_ptr()
        a.states, a.actions, a.rewards, a.phis, a.next_states, a.gammas = (t.data_ptr() for t in self._out)

    def append(self, state, action, reward, phi, next_state, gamma):
        """
        One transition -> one packed fp32 row of the ring.  Host-resident fields (what the environments hand over) are
        assembled into a pinned staging row and leave with ONE asynchronous copy: no device sync, no per-field launches
        (the reference stores python tuples, sfdqn.py:86-89).  Device-resident fields fall back to a device-side concatenation.
        """
        parts = (state, next_state, phi, reward, gamma, action)
        if any(torch.is_tensor(v) and v.is_cuda for v in parts):
            dev = _device()
            flat = lambda v: torch.as_tensor(v).detach().to(dev, non_blocking=True).to(torch.float32).reshape(-1)
            row = torch.cat([flat(v) for v in parts])
            if self.ring is None:
                self._alloc(flat(state).numel(), flat(phi).numel())
            self.ring[self.index].copy_(row)
        else:
            host = [np.asarray(v.detach() if torch.is_tensor(v) else v, dtype=np.float32).reshape(-1) for v in parts]
            if host[5][0] >= (1 << 24):
                raise ValueError('action index too large for the packed fp32 row')
            if self.ring is None:
                self._alloc(host[0].size, host[2].size)
            k = self._row_slot = (self._row_slot + 1) % len(self._row_host)
            if self._row_done[k] is not None:
                self._row_done[k].synchronize()              # (waits only when the host is a whole staging ring ahead)
            np.concatenate(host, out=self._row_host[k].numpy())
            self.ring[self.index].copy_(self._row_host[k], non_blocking=True)
            ev = self._row_done[k] = self._row_done[k] or torch.cuda.Event()
            ev.record()
        self.size = min(self.size + 1, self.n_samples)
        self.index = (self.index + 1) % self.n_samples

    def replay(self):
        """None until n_batch samples exist (sfdqn.py:57); else (states, actions, rewards, phis, next_states, gammas)."""
        if self.size < self.n_batch:
            return None
        import ctypes as C
        from . import _lib
        k = self._picks_slot = (self._picks_slot + 1) % len(self._picks_host)
        if self._picks_done[k] is not None:
            self._picks_done[k].synchronize()                # (only ever waits when the host is > 3 replays ahead)
        self._picks_host[k].copy_(torch.from_numpy(np.random.randint(low=0, high=self.size, size=(self.n_batch,))))
        self._picks.copy_(self._picks_host[k], non_blocking=True)
        ev = self._picks_done[k] = self._picks_done[k] or torch.cuda.Event()
        ev.record()
        _lib.call('sfgpi_replay_gather', C.byref(self._args), C.c_void_p(torch.cuda.current_stream().cuda_stream))
        return self._out

    def state_dict(self):
        """ReplayBuffer.state_dict()'s format: clones of the packed rows [:size], split into fields (fp32, actions int64)."""
        n, sd = self.size, dict(n_samples=self.n_samples, index=self.index, size=self.size)
        if self.ring is None:
            return dict(sd, **{k: torch.empty(0) for k in _RING_FIELDS})
        S, D, rows = self.S, self.D, self.ring[:n]
        return dict(sd, states=rows[:, :S].clone(), next_states=rows[:, S:2 * S].clone(), phis=rows[:, 2 * S:2 * S + D].clone(),
                    rewards=rows[:, 2 * S + D].clone(), gammas=rows[:, 2 * S + D + 1].clone(),
                    actions=rows[:, 2 * S + D + 2].to(torch.int64))

    def load_state_dict(self, sd):
        _check_ring_dict(self, sd)
        self.reset()
        n = int(sd['size'])
        if n:
            dev = _device()
            col = lambda k: sd[k].detach().to(device=dev, dtype=torch.float32).reshape(n, -1)
            S, D = col('states').shape[1], col('phis').shape[1]
            if int(sd['actions'].max()) >= (1 << 24):
                raise ValueError('action index too large for the packed fp32 row')
            self._alloc(S, D)
            self.ring[:n].copy_(torch.cat([col(k) for k in ('states', 'next_states', 'phis', 'rewards', 'gammas', 'actions')], 1))
        self.index, self.size = int(sd['index']), n


class PackedPsi(torch.nn.Module):
    """
    The per-task psi module handed to callers in `sf.psi[i]`.  Its Linear parameters are views of row i of the packed
    library, so parameters()/state_dict()/update_models_weights work; calling it runs the fused CUDA forward.
    """

    def __init__(self, net, library, index, target):
        super().__init__()
        self.net = net
        self._lib_ref = [library]          # list: keep the library out of the module tree
        self.index, self.is_target = index, target

    def forward(self, state):
        lib = self._lib_ref[0]
        if lib.autograd and not self.is_target and torch.is_grad_enabled():
            return lib.psi(state, self.index, 1)[:, 0]
        return lib.forward_psi(state, self.index, 1, target=self.is_target)[:, 0]


class PackedAdamView:
    """
    Optimizer i's Adam in the packed buffers, shaped like torch.optim.Adam's `state` / `param_groups`.  The fused train step
    steps it inside update_successor.  On a library built with autograd=True, step() / zero_grad() also work the reference's
    eager way (optim.zero_grad(); loss.backward(); optim.step()): one sfgpi_adam_step launch over the groups that have
    gradients -- the psi row from the packed gradient online.grad[i], w, and for TSF g and the shared h -- sharing `step`
    and the bias corrections with the fused step, so both kinds of step can be mixed.
    """

    def __init__(self, library, index, groups, eager_unsupported=None):
        self._library, self.index, self._groups = library, index, groups
        self._eager_unsupported = eager_unsupported
        self._skipped = set()        # groups left out of an eager step while others were stepped

    @property
    def param_groups(self):
        L = self._library
        return [dict(params=p, lr=L.lr[k], weight_decay=L.wd[k], betas=(0.9, 0.999), eps=1e-8) for k, p in self._groups]

    _MOMENTS = {'sf': ('m', 'v'), 'w': ('w_m', 'w_v'), 'g': ('g_m', 'g_v'), 'h': ('h_m', 'h_v')}

    def _moments(self, src, row=None):
        """[(param, exp_avg, exp_avg_sq)] in param-id order: views of row `row` (default i) of the moment buffers src(name) (the
        library's, or those of its state_dict), at each parameter's offset into its packed row."""
        L, i, out = self._library, self.index, []
        base = {'sf': L.online.detach()[i], 'w': L.w[i], 'h': L.h, 'g': L.g[i] if L.G is not None else None}
        for k, params in self._groups:
            m, v = (src(name)[i if row is None else row] for name in self._MOMENTS[k])
            for p in params:
                off = (p.data.data_ptr() - base[k].data_ptr()) // 4
                out.append((p, m[off:off + p.numel()].view_as(p), v[off:off + p.numel()].view_as(p)))
        return out

    @property
    def state(self):
        L = self._library
        step = L.step[self.index]
        return {p: dict(step=step, exp_avg=m, exp_avg_sq=v) for p, m, v in self._moments(lambda name: getattr(L, name))}

    def state_dict(self):
        """torch.optim.Adam.state_dict() of optimizer i: one param group per kind in the reference's order (psi, w, and for TSF
        g's W and b, h's W and b), integer param ids, and per parameter a 0-dim float32 `step` with clones of its moments (no
        state before the first step).  Loads into a stock torch.optim.Adam over the same parameters, and back."""
        L = self._library
        return self._torch_dict(lambda name: getattr(L, name), int(L.step[self.index]), clone=True)

    def _torch_dict(self, src, step, clone=False, row=None):
        state = {}
        if step > 0:
            for pid, (_, m, v) in enumerate(self._moments(src, row)):
                state[pid] = dict(step=torch.tensor(float(step)), exp_avg=m.clone() if clone else m,
                                  exp_avg_sq=v.clone() if clone else v)
        groups, pid = [], 0
        for g in self.param_groups:
            n = len(g['params'])
            groups.append(dict(g, amsgrad=False, maximize=False, params=list(range(pid, pid + n))))
            pid += n
        return dict(state=state, param_groups=groups)

    def load_state_dict(self, sd):
        """Load a torch.optim.Adam.state_dict() over the same parameters (or this class's own): the moments go into the packed
        rows at the parameters' offsets.  Each group's lr / weight decay must be the library's, which steps every optimizer's
        group of that kind alike.  The packed step counter is one per optimizer, so every parameter with state must carry the
        same step; parameters without state are allowed only when no parameter has any (a fresh optimizer)."""
        L, i = self._library, self.index
        groups = sd['param_groups']
        if [len(g['params']) for g in groups] != [len(p) for _, p in self._groups]:
            raise ValueError(f'optimizer {i}: the state_dict\'s parameter groups {[len(g["params"]) for g in groups]} do not '
                             f'match this optimizer\'s {[len(p) for _, p in self._groups]}')
        for (k, _), g in zip(self._groups, groups):
            if tuple(g.get('betas', (ADAM_BETA1, ADAM_BETA2))) != (ADAM_BETA1, ADAM_BETA2) or g.get('eps', ADAM_EPS) != ADAM_EPS \
                    or g.get('amsgrad', False) or g.get('maximize', False):
                raise ValueError(f'optimizer {i}: the packed Adam runs betas=(0.9, 0.999), eps=1e-8 without amsgrad / maximize')
            if g['lr'] != L.lr[k] or g.get('weight_decay', 0.0) != L.wd[k]:
                raise ValueError(f"optimizer {i}: group '{k}' has lr={g['lr']}, weight_decay={g.get('weight_decay', 0.0)}; the "
                                 f"library steps every optimizer's '{k}' group with lr={L.lr[k]}, weight_decay={L.wd[k]}")
        ids = [pid for g in groups for pid in g['params']]
        have = [pid in sd['state'] for pid in ids]
        if any(have) and not all(have):
            raise ValueError(f'optimizer {i}: only some parameters have Adam state; the packed step counter is one per optimizer')
        steps = {float(sd['state'][pid]['step']) for pid in ids} if all(have) else {0.0}
        if len(steps) != 1:
            raise ValueError(f'optimizer {i}: the parameters carry different Adam steps {sorted(steps)}; the packed step counter '
                             'is one per optimizer')
        step = steps.pop()
        with torch.no_grad():
            for pid, (p, m, v) in zip(ids, self._moments(lambda name: getattr(L, name))):
                st = sd['state'].get(pid)
                m.copy_(st['exp_avg'] if st is not None else torch.zeros_like(m))
                v.copy_(st['exp_avg_sq'] if st is not None else torch.zeros_like(v))
            L.step[i] = int(step)
        L._refresh_adam(i, 1)
        self._skipped = set()

    def zero_grad(self, set_to_none=True):
        """Clears optimizer i's psi row of the packed gradient and the .grad of every parameter it steps (w, g and the
        shared h included, as torch.optim.Adam.zero_grad does for its groups)."""
        L = self._library
        if not L.autograd:
            return
        i = self.index
        if L.online.grad is not None:
            L.online.grad[i].zero_()
        L._grad_rows.discard(i)
        L._bound_rows.discard(i)
        for _, params in self._groups:
            for p in params:
                if p.grad is None:
                    continue
                if set_to_none:
                    p.grad = None
                else:
                    p.grad.detach_().zero_()

    def step(self):
        L, i = self._library, self.index
        if not L.autograd:
            raise RuntimeError('the packed Adam is stepped inside update_successor (fused kernel); it has no standalone step()')
        if self._eager_unsupported is not None or L.n_flows > 0:
            raise NotImplementedError(f'optim.step() is not supported for {self._eager_unsupported or "normalising-flow g functions"}; '
                                      'use the fused update_successor')
        if L._sharded:
            raise NotImplementedError('optim.step() does not support sharded libraries')
        have = {}
        for k, params in self._groups:
            n_grad = sum(p.grad is not None for p in params)
            if 0 < n_grad < len(params):
                raise RuntimeError(f"optimizer {i}: only some parameters of the '{k}' group have gradients; the packed Adam "
                                   'steps a group as a whole')
            have[k] = n_grad > 0
        have.setdefault('g', False)
        have.setdefault('h', False)
        for k in self._skipped:
            if have[k]:
                raise RuntimeError(f"optimizer {i}: the '{k}' group was skipped by an earlier step and now has gradients; the "
                                   'packed per-optimizer step counter cannot represent a per-parameter step')
        if not any(have.values()):
            return
        self._skipped |= {k for k, h in have.items() if not h}
        self._launch(have)

    def _launch(self, have):
        import ctypes as C
        from . import _lib
        from .library import AdamSeg, _stream, adam_args
        L, i = self._library, self.index
        sp = L.spec
        keep = []                                    # tensors that must outlive the launch call

        def grad_of(p):
            g = p.grad.detach()
            if g.dtype != torch.float32 or not g.is_contiguous() or g.device != L.device:
                g = g.to(device=L.device, dtype=torch.float32).contiguous()
            keep.append(g)
            return g.data_ptr()

        segs = []
        if have['sf']:
            row = L.online.grad[i]
            for (W, b), lin in zip(sp.views(row), L._views[i]['online']):      # .grad rebound by the user: copy it back
                for view, p in ((W, lin.weight), (b, lin.bias)):
                    if p.grad.data_ptr() != view.data_ptr():
                        view.copy_(p.grad)
            segs.append(AdamSeg(L.online.detach()[i].data_ptr(), L.m[i].data_ptr(), L.v[i].data_ptr(), row.data_ptr(), sp.row_stride,
                                L.lr['sf'], L.wd['sf']))
        if have['w']:
            segs.append(AdamSeg(L.w[i].data_ptr(), L.w_m[i].data_ptr(), L.w_v[i].data_ptr(), grad_of(self._groups[1][1][0]),
                                sp.n_features, L.lr['w'], L.wd['w']))
        if L.G is not None:
            S, G, D = sp.dims[0], L.G, sp.n_features
            if have['g']:
                gW, gb = self._groups[2][1]
                p, m, v, o = L.g[i].data_ptr(), L.g_m[i].data_ptr(), L.g_v[i].data_ptr(), 4 * G * S
                segs.append(AdamSeg(p, m, v, grad_of(gW), G * S, L.lr['g'], L.wd['g']))
                segs.append(AdamSeg(p + o, m + o, v + o, grad_of(gb), G, L.lr['g'], L.wd['g']))
            if have['h']:
                hW, hb = self._groups[3][1]
                p, m, v, o = L.h.data_ptr(), L.h_m[i].data_ptr(), L.h_v[i].data_ptr(), 4 * D * G
                segs.append(AdamSeg(p, m, v, grad_of(hW), D * G, L.lr['h'], L.wd['h']))
                segs.append(AdamSeg(p + o, m + o, v + o, grad_of(hb), D, L.lr['h'], L.wd['h']))
        # bias corrections: the same double-buffered pair the fused step reads and advances (library.train_step)
        ad = adam_args(segs, 1, L.step[i:].data_ptr(), L._adam_consts(i, 1))
        _lib.call('sfgpi_adam_step', C.byref(ad), _stream())
        L.weights_gen += 1


class DeepSF:
    """Successor-feature library, G2 ("sequential") semantics  [sfdqn.py:94-371]."""

    _eager_step_unsupported = None

    def __init__(self, pytorch_model_handle, use_true_reward=False, target_update_ev=1000, **kwargs):
        self.use_true_reward = use_true_reward
        self.hyperparameters = kwargs.get('hyperparameters', {})
        self.alpha_w = self.hyperparameters.get('learning_rate_w')
        self.pytorch_model_handle = pytorch_model_handle
        self.target_update_ev = target_update_ev
        self.device = _device()
        self._tsf_dim = None
        self._library = None
        self.precision = kwargs.get('precision', self.hyperparameters.get('precision', 'fp32'))
        # autograd=True: get_successor(s) and the online psi modules record a differentiable forward under grad mode, and the
        # optimizers' step() / zero_grad() work, so the reference's eager update code runs on the packed library
        self.autograd = bool(kwargs.get('autograd', self.hyperparameters.get('autograd', False)))
        # state_grad=True (needs autograd): those forwards also take states that require grad and pass dL/dstate back, e.g. to a
        # learned state encoder in front of psi.  Target nets stay constants: they raise for such states under grad mode.
        # GPI / GPI_w / greedy_action are not differentiable.
        self.state_grad = bool(kwargs.get('state_grad', self.hyperparameters.get('state_grad', False)))
        if self.state_grad and not self.autograd:
            raise ValueError('state_grad=True needs autograd=True')

    # ---- library construction -------------------------------------------------------------------------------------
    def _hyper(self, kind, default):
        return {k: self.hyperparameters.get(f'{kind}_{k}', default) for k in ('sf', 'w', 'g', 'h')}

    def _new_library(self):
        lr, wd = self._hyper('learning_rate', 1e-3), self._hyper('weight_decay', 0.0)
        return PackedSFLibrary(self.device, lr=lr, wd=wd, tsf_dim=self._tsf_dim, precision=self.precision, autograd=self.autograd,
                               state_grad=self.state_grad)

    def reset(self):
        self.n_tasks = 0
        self.psi = []
        self.true_w = []
        self.fit_w = []
        self.gpi_counters = []
        self.updates_since_target_updated = []
        self._library = self._new_library()

    def GPI_usage_percent(self, task_index):
        counts = self.gpi_counters[task_index]
        return 1. - (float(counts[task_index]) / np.sum(counts))

    def add_training_task(self, task, source=None):
        true_w = task.get_w()
        n_features = task.feature_dim()
        w_approx = torch.nn.Linear(n_features, 1, bias=False, device=self.device)
        with torch.no_grad():
            w_approx.weight.uniform_(-0.01, 0.01)                       # sfdqn.py:197
        self.true_w.append(true_w)
        self.fit_w.append(w_approx)
        self.psi.append(self.build_successor(task, source, w_approx))
        self.n_tasks = len(self.psi)
        for i in range(len(self.gpi_counters)):
            self.gpi_counters[i] = np.append(self.gpi_counters[i], 0)
        self.gpi_counters.append(np.zeros((self.n_tasks,), dtype=int))

    def build_successor(self, task, source=None, w_approx=None, g_function=None, h_function=None):
        if self.n_tasks == 0:
            self.n_actions = task.action_count()
            self.n_features = task.feature_dim()
            self.inputs = task.encode_dim()
        shape = (self.inputs, self.n_actions * self.n_features, (self.n_actions, self.n_features), 1)
        model, loss, _ = self.pytorch_model_handle(*shape)
        target_model, _, _ = self.pytorch_model_handle(*shape)
        with torch.no_grad():
            if source is not None and self.n_tasks > 0:                  # warm start from a source policy (sfdqn.py:255-259)
                src = self.psi[source][0][0].net
                for p_new, p_src in zip(model.parameters(), src.parameters()):
                    p_new.copy_(p_src)
            for p_t, p in zip(target_model.parameters(), model.parameters()):
                p_t.copy_(p)                                             # target <- online at construction
        index = self._library.add_policy(model, target_model, w_approx, g_function, h_function, self.n_actions, self.n_features)
        self.updates_since_target_updated.append(0)
        online = PackedPsi(model, self._library, index, target=False)
        target = PackedPsi(target_model, self._library, index, target=True)
        target.eval()
        groups = [('sf', list(model.parameters())), ('w', list(w_approx.parameters()))]
        if g_function is not None:
            groups += [('g', list(g_function.parameters())), ('h', list(h_function.parameters()))]
        optim = PackedAdamView(self._library, index, groups, eager_unsupported=self._eager_step_unsupported)
        return (online, loss, optim), (target, None, None)

    # ---- forwards ---------------------------------------------------------------------------------------------------
    def get_successor(self, state, policy_index):
        if self.autograd and torch.is_grad_enabled():
            return self._library.psi(state, policy_index, 1)[:, 0]
        return self._library.forward_psi(state, policy_index, 1)[:, 0]

    def get_successors(self, state):
        if self.autograd and torch.is_grad_enabled():
            return self._library.psi(state, 0, self.n_tasks)
        return self._library.forward_psi(state, 0, self.n_tasks)

    # ---- GPI ----------------------------------------------------------------------------------------------------------
    def GPI_w(self, state, w):
        """q [n_batch, n_tasks, n_actions] and the task active in GPI per state (squeezed, sfdqn.py:239).  Not differentiable,
        with autograd / state_grad too: q carries no gradient to psi, w or the states."""
        w_vec = w.weight if isinstance(w, torch.nn.Module) else w
        q, _, key_task = self._library.gpi(state, w_vec)
        task = torch.squeeze(self._library.decode_keys(key_task))
        return q, task

    def GPI(self, state, task_index, update_counters=False):
        q, task = self.GPI_w(state, self.fit_w[task_index])
        if update_counters:
            self.gpi_counters[task_index][task.cpu().numpy()] += 1
        return q, task

    def greedy_action(self, state, task_index, use_gpi=True, agent=None):
        """
        The action-selection call of next_sample (sfdqn.py:585-594 / tsfdqn.py:529-535, 420-433) in one fused pass: GPI under
        fit_w[task_index], c = argmax_j max_a q (counted in gpi_counters when use_gpi, as GPI(update_counters=True) does),
        a = argmax_a q[0, c, :].  use_gpi=False: c = task_index and only that policy's net runs.  One device->host read of
        (a, c) -- the same single sync the reference pays at `int(action)` (tasks/reacher.py:46).  Returns a 0-dim int64 tensor.
        """
        lib = self._library
        w = self.fit_w[task_index]
        w_vec = w.weight if isinstance(w, torch.nn.Module) else w
        if use_gpi:
            idx = lib.gpi_select(state, w_vec)
        else:
            idx = lib.gpi_select(state, w_vec, task_index, 1)
        if idx.shape[1] != 1:
            raise ValueError('greedy_action selects for ONE state (the agents act at batch 1)')
        a, c = (int(v) for v in idx[:, 0].tolist())
        if not use_gpi:
            c = task_index
        else:
            self.gpi_counters[task_index][c] += 1
        if agent is not None:
            agent.c = c
        return torch.tensor(a)

    # ---- train step ---------------------------------------------------------------------------------------------------
    def _after_update(self, policy_index):
        self.updates_since_target_updated[policy_index] += 1
        if self.updates_since_target_updated[policy_index] >= self.target_update_ev:
            self._library.target_sync(policy_index)
            self.updates_since_target_updated[policy_index] = 0

    def update_successor(self, transitions, policy_index, use_gpi=True):
        if transitions is None:
            return
        losses = self._library.train_step(transitions, policy_index, use_gpi=use_gpi, variant=1)
        self._after_update(policy_index)
        return losses[0, 0], losses[0, 1], losses[0, 2]

    def update_successor_all(self, transitions, use_gpi=True):
        """Ensemble extension: every policy stepped on the same batch in one fused pass (frozen-snapshot semantics)."""
        if transitions is None:
            return
        losses = self._library.train_step(transitions, 'all', use_gpi=use_gpi, variant=1)
        for i in range(self.n_tasks):
            self._after_update(i)
        return losses

    # ---- checkpoints --------------------------------------------------------------------------------------------------
    def state_dict(self):
        """
        Training state of the library: sd['library'] (PackedSFLibrary.state_dict: every network, reward vector, g / h and Adam
        state) with gpi_counters, updates_since_target_updated, n_tasks and target_update_ev.  sd['library'] is the source of
        truth.  sd['psi'][i] = {'model': ..., 'optim': ...} is task i in the layout of the reference's eager objects --
        psi_model.state_dict() key names and torch.optim.Adam.state_dict() -- built from VIEWS of sd['library']'s tensors, so
        torch.save stores the data once; load it into a reference psi_model / torch.optim.Adam to continue task i eagerly.
        load_state_dict reads sd['library'] only.  Everything a TSF library learns (g, h) lives in the library too.

        On a policy-sharded library this is a collective over the shard's process group (PackedSFLibrary.state_dict): every
        rank returns the same dict of ALL the group's tasks in global task order -- the format of one unsharded library
        holding them, loadable at any GPU count.  GPI selects global task indices, so a gpi_counters row holds one count per
        global task; rows shorter than that (built before the library was sharded) are padded with zeros.
        """
        lib = self._library
        lsd = lib.state_dict()
        lo, n_total = self._task_range()
        counters = [np.asarray(c).tolist() for c in self.gpi_counters]
        updates = list(self.updates_since_target_updated)
        if lib._sharded:
            import torch.distributed as dist
            parts = [None] * lib.shard.world
            dist.all_gather_object(parts, (counters, updates), group=lib.shard.group)
            counters, updates = [c for p in parts for c in p[0]], [u for p in parts for u in p[1]]
        counters = [c + [0] * (n_total - len(c)) for c in counters]
        psi = []
        for i in range(n_total):
            k = i - lo if lo <= i < lo + self.n_tasks else 0    # another rank's task: task 0's modules (one architecture)
            (model, _, optim), _ = self.psi[k]
            names = {p: n for n, p in model.net.named_parameters()}
            weights = OrderedDict()
            for (W, b), lin in zip(lib.spec.views(lsd['online'][i]), lib._views[k]['online']):
                weights[names[lin.weight]], weights[names[lin.bias]] = W, b
            psi.append(dict(model=weights, optim=optim._torch_dict(lsd.__getitem__, int(lsd['step'][i]), row=i)))
        return dict(library=lsd, psi=psi, gpi_counters=counters, updates_since_target_updated=updates, n_tasks=n_total,
                    target_update_ev=self.target_update_ev)

    def load_state_dict(self, sd):
        """Restore a state_dict() into a library that already holds the same tasks (add them first, as the saved run did).
        On a policy-sharded library every rank passes the same full dict of all the group's tasks and keeps its own."""
        for k in ('library', 'gpi_counters', 'updates_since_target_updated', 'n_tasks', 'target_update_ev'):
            if k not in sd:
                raise ValueError(f"SF state_dict: missing key '{k}'")
        lo, n_total = self._task_range()
        if sd['n_tasks'] != n_total:
            raise ValueError(f"SF state_dict: it holds {sd['n_tasks']} tasks, this library holds {n_total}")
        self._library.load_state_dict(sd['library'])
        mine = slice(lo, lo + self.n_tasks)
        self.gpi_counters = [np.asarray(c, dtype=int) for c in sd['gpi_counters'][mine]]
        self.updates_since_target_updated = list(sd['updates_since_target_updated'][mine])
        self.target_update_ev = sd['target_update_ev']

    def _task_range(self):
        """(lo, n_total): this object's tasks are tasks [lo, lo + n_tasks) of the n_total of its library's shard group
        ((0, n_tasks) unsharded)."""
        lib = self._library
        return (lib.shard.lo, lib.shard.n_total) if lib._sharded else (0, self.n_tasks)


class SFDQN:
    """SFDQN agent, sequential variant  [sfdqn.py:374-749].  Host-side RL loop around the fused SF library."""

    def __init__(self, deep_sf, buffer_handle, gamma, T, encoding, epsilon=0.1, epsilon_decay=1, epsilon_min=0, print_ev=1000,
                 save_ev=100, use_gpi=True, test_epsilon=0.03, **kwargs):
        self.gamma, self.T = gamma, T
        self.encoding = (lambda s: s) if encoding is None else encoding
        self.epsilon_init, self.epsilon_decay, self.epsilon_min = epsilon, epsilon_decay, epsilon_min
        self.print_ev, self.save_ev = print_ev, save_ev
        self.total_training_steps = 0
        self.sf = deep_sf
        self.buffer_handle = buffer_handle
        self.use_gpi = use_gpi
        self.test_epsilon = test_epsilon
        self.logger = kwargs.get('logger', None)
        self.test_tasks_weights = []
        self.hyperparameters = kwargs.get('hyperparameters', {})
        self.buffers = []
        self.device = _device()

    # ---- task management ----------------------------------------------------------------------------------------------
    def reset(self):
        self.tasks, self.phis = [], []
        self.cum_reward, self.reward_hist, self.cum_reward_hist = 0., [], []
        self.sf.reset()
        for buffer in self.buffers:
            buffer.reset()

    def add_training_task(self, task):
        self.tasks.append(task)
        self.n_tasks = len(self.tasks)
        self.phis.append(task.features)
        if self.n_tasks == 1:
            self.n_actions = task.action_count()
            self.n_features = task.feature_dim()
            if self.encoding == 'task':
                self.encoding = task.encode
        self.sf.add_training_task(task, source=None)
        self.buffers.append(self.buffer_handle())

    def set_active_training_task(self, index):
        self.task_index = index
        self.active_task = self.tasks[index]
        self.phi = self.phis[index]
        self.s = self.s_enc = None
        self.new_episode = True
        self.episode, self.episode_reward = 0, 0.
        self.steps_since_last_episode, self.reward_since_last_episode = 0, 0.
        self.steps, self.reward = 0, 0.
        self.epsilon = self.epsilon_init
        self.episode_reward_hist = []
        self.buffer = self.buffers[index]

    # ---- the two L3-facing calls ----------------------------------------------------------------------------------------
    def train_agent(self, s, s_enc, a, r, s1, s1_enc, gamma):
        phi = self.phi(s, a, s1)
        self.buffer.append(s_enc, a, r, phi, s1_enc, gamma)
        transitions = self.buffer.replay()
        losses = self.sf.update_successor(transitions, self.task_index, self.use_gpi)
        if isinstance(losses, tuple) and self.logger is not None:
            total_loss, psi_loss, phi_loss = losses
            self.logger.log_losses(total_loss.item(), psi_loss.item(), phi_loss.item(), [1], self.total_training_steps)

    def _greedy_action(self):
        """sfdqn.py:585-594: a = argmax_a q[0, c, :], c = the GPI task (use_gpi) or the active task -- read off the packed keys."""
        return self.sf.greedy_action(self.s_enc, self.task_index, self.use_gpi, agent=self)

    def _choose_action(self):
        """epsilon-greedy of sfdqn.py:578-597: the GPI forward runs (and the GPI counters move) only on greedy steps."""
        if random.random() <= self.epsilon:
            a = torch.tensor(random.randrange(self.n_actions))
        else:
            a = self._greedy_action()
        self.epsilon = max(self.epsilon * self.epsilon_decay, self.epsilon_min)
        return a

    def next_sample(self, viewer=None, n_view_ev=None):
        if self.new_episode:
            self.s = self.active_task.initialize()
            self.s_enc = self.encoding(self.s)
            self.new_episode = False
            self.episode += 1
            self.steps_since_last_episode = 0
            self.episode_reward = self.reward_since_last_episode
            self.reward_since_last_episode = 0.
            if self.episode > 1:
                self.episode_reward_hist.append(self.episode_reward)
        a = self._choose_action()
        s1, r, terminal = self.active_task.transition(a)
        s1_enc = self.encoding(s1)
        gamma = 0. if terminal else self.gamma
        if terminal:
            self.new_episode = True
        self.train_agent(self.s, self.s_enc, a, r, s1, s1_enc, gamma)
        self.s, self.s_enc = s1, s1_enc
        self.steps += 1
        self.reward += r
        self.steps_since_last_episode += 1
        self.reward_since_last_episode += r
        self.cum_reward += r
        if self.steps_since_last_episode >= self.T:
            self.new_episode = True
        if self.steps % self.save_ev == 0:
            self.reward_hist.append(self.reward)
            self.cum_reward_hist.append(self.cum_reward)
        if viewer is not None and self.episode % n_view_ev == 0:
            viewer.update()

    def get_progress_dict(self):
        gpi_percent = self.sf.GPI_usage_percent(self.task_index)
        w_error = torch.linalg.norm(self.sf.fit_w[self.task_index].weight.T - torch.as_tensor(self.sf.true_w[self.task_index]).to(self.device))
        return {'task': self.task_index, 'steps': self.total_training_steps, 'episodes': self.episode, 'eps': self.epsilon,
                'ep_reward': self.episode_reward, 'reward': self.reward, 'reward_hist': self.reward_hist,
                'cum_reward': self.cum_reward, 'cum_reward_hist': self.cum_reward_hist, 'GPI%': gpi_percent, 'w_err': w_error}

    def train(self, train_tasks, n_samples, viewers=None, n_view_ev=None, test_tasks=[], n_test_ev=1000, cycles_per_task=1):
        if viewers is None:
            viewers = [None] * len(train_tasks)
        self.reset()
        for train_task in train_tasks:
            self.add_training_task(train_task)
        for test_task in test_tasks:
            self.test_tasks_weights.append(self._new_test_task(test_task.feature_dim()))
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
                    self.total_training_steps += 1
        return return_data

    # ---- checkpoints --------------------------------------------------------------------------------------------------
    _EPISODE = ('s', 's_enc', 'new_episode', 'episode', 'episode_reward', 'steps_since_last_episode', 'reward_since_last_episode',
                'steps', 'reward', 'episode_reward_hist', 'cum_reward', 'reward_hist', 'cum_reward_hist')

    def state_dict(self):
        """
        Training state of the agent: the SF library's state_dict, every task's replay ring, total_training_steps, epsilon, the
        active task with its episode in progress, and the target tasks' reward vectors with their optimizers.  As in torch, the
        random streams (Python `random`, numpy, torch) and the environments' own state are the caller's to save and restore.
        """
        self._check_unsharded('state_dict')
        active = getattr(self, 'task_index', None)
        return dict(sf=self.sf.state_dict(), buffers=[b.state_dict() for b in self.buffers],
                    total_training_steps=self.total_training_steps, epsilon=getattr(self, 'epsilon', self.epsilon_init),
                    task_index=active, episode={k: list(v) if isinstance(v, list) else v
                                                for k, v in vars(self).items() if k in self._EPISODE},
                    test_tasks=[self._test_task_state(k) for k in range(len(self.test_tasks_weights))])

    def load_state_dict(self, sd):
        """Restore a state_dict() into an agent that already holds the same training tasks (reset() + add_training_task, as
        the saved run did).  Target tasks are rebuilt when the agent has none yet."""
        self._check_unsharded('load_state_dict')
        if len(sd['buffers']) != len(self.buffers):
            raise ValueError(f"agent state_dict: it holds {len(sd['buffers'])} tasks, this agent holds {len(self.buffers)}")
        if self.test_tasks_weights and len(self.test_tasks_weights) != len(sd['test_tasks']):
            raise ValueError(f"agent state_dict: it holds {len(sd['test_tasks'])} target tasks, this agent holds "
                             f"{len(self.test_tasks_weights)}")
        self.sf.load_state_dict(sd['sf'])
        for buf, bsd in zip(self.buffers, sd['buffers']):
            buf.load_state_dict(bsd)
        self.total_training_steps = sd['total_training_steps']
        if sd['task_index'] is not None:
            self.set_active_training_task(sd['task_index'])
            for k, v in sd['episode'].items():
                setattr(self, k, list(v) if isinstance(v, list) else v)
        self.epsilon = sd['epsilon']
        for k, tsd in enumerate(sd['test_tasks']):
            self._load_test_task(k, tsd)

    def _check_unsharded(self, what):
        lib = getattr(self.sf, '_library', None)
        if lib is not None and lib._sharded:
            raise NotImplementedError(f'{type(self).__name__}.{what}() does not support policy-sharded libraries: the replay '
                                      'rings are per rank.  Save and load the SF library with sf.state_dict() / '
                                      'sf.load_state_dict(), collectively on every rank')

    def _new_test_task(self, feature_dim):
        """(w_approx, torch.optim.Adam over it) of one target task, as train() builds them."""
        w_approx = torch.nn.Linear(feature_dim, 1, bias=False, device=self.device)
        with torch.no_grad():
            w_approx.weight.uniform_(-0.01, 0.01)
        optim = torch.optim.Adam([{'params': w_approx.parameters(), 'lr': self.hyperparameters['learning_rate_w'],
                                   'weight_decay': self.hyperparameters['weight_decay_w']}])
        return w_approx, optim

    def _test_task_state(self, k):
        w, optim = self.test_tasks_weights[k]
        return dict(w=w.weight.detach().clone(), optim=optim.state_dict())

    def _load_test_task(self, k, tsd):
        if k == len(self.test_tasks_weights):
            self.test_tasks_weights.append(self._new_test_task(tsd['w'].numel()))
        w, optim = self.test_tasks_weights[k]
        with torch.no_grad():
            w.weight.copy_(tsd['w'].reshape(w.weight.shape))
        optim.load_state_dict(tsd['optim'])

    # ---- target tasks (host loop; calls the in-scope get_successors) -----------------------------------------------------
    def get_test_action(self, s_enc, w):
        with torch.no_grad():
            if random.random() <= self.test_epsilon:
                return torch.tensor(random.randrange(self.n_actions)).to(self.device)
            q, task = self.sf.GPI_w(s_enc, w)
            return torch.argmax(q[:, task, :])

    def test_agent(self, task, test_index):
        R = 0.0
        w, optim = self.test_tasks_weights[test_index]
        s = task.initialize()
        s_enc = self.encoding(s)
        for _ in range(self.T):
            a = self.get_test_action(s_enc, w)
            s1, r, done = task.transition(a)
            s1_enc = self.encoding(s1)
            self.update_test_reward_mapper(w, optim, task, r, s_enc, a, s1_enc)
            s, s_enc = s1, s1_enc
            R += r
            if done:
                break
        return R

    def update_test_reward_mapper(self, w_approx, optim, task, r, s, a, s1):
        phi = torch.as_tensor(task.features(s, a, s1)).float().to(self.device)
        r_tensor = torch.tensor(r).float().unsqueeze(0).to(self.device)
        optim.zero_grad()
        loss = torch.nn.functional.mse_loss(w_approx(phi), r_tensor)
        loss.backward()
        optim.step()
        return loss
