# -*- coding: UTF-8 -*-
"""
PackedSFLibrary: HBM-resident storage + kernel orchestration for an ensemble of N successor-feature networks.

Replaces the reference's per-task Python objects -- N `nn.Sequential` psi nets + N target copies + N `nn.Linear` reward
maps + N `torch.optim.Adam` (sfdqn.py:180-288, tsfdqn.py:137-281) -- by a handful of packed fp32 buffers

    online / target / exp_avg / exp_avg_sq : [cap][row_stride]      one row per policy (layout: include/sfgpi.h)
    w, w_m, w_v                            : [cap][D]
    g, g_m, g_v                            : [cap][G*S + G]          (TSF g_i: Linear(S,G), tsfdqn.py:537)
    h : [D*G + D] shared;  h_m, h_v        : [cap][D*G + D]          (one Adam state per policy-optimizer, tsfdqn.py:255-270)
    step                                   : [cap] int32 (device)    Adam step counters

and runs every reference hot-path function through the C ABI (libsfgpi.so).  The per-task `nn.Module` objects handed back to
the agents hold VIEWS of row i, so `.parameters()`, `state_dict()`, `update_models_weights` and `fit_w[i].weight` keep
working.  No torch op is on the compute path; torch only owns the memory and the stream.
"""
import ctypes as C
import math

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from . import _lib
from ._lib import ACT, MAX_LAYERS, ptr

INT64_MIN = -(1 << 63)


class NetSpec:
    """Shape of one psi network, adopted from the `nn.Sequential` that `pytorch_model_handle` returns."""

    def __init__(self, dims, acts, n_actions, n_features):
        assert len(acts) == len(dims) - 1
        if len(acts) > MAX_LAYERS:
            raise ValueError(f'at most {MAX_LAYERS} Linear layers are supported')
        if dims[-1] != n_actions * n_features:
            raise ValueError('psi output width must be n_actions * n_features')
        if acts[-1] != 'none':
            raise ValueError('the psi output layer must be linear (no activation)')
        self.dims, self.acts = list(dims), list(acts)
        self.n_actions, self.n_features = n_actions, n_features
        off, self.w_off, self.b_off = 0, [], []
        for l in range(len(acts)):
            self.w_off.append(off)
            off += (dims[l + 1] * dims[l] + 3) & ~3
            self.b_off.append(off)
            off += (dims[l + 1] + 3) & ~3
        self.n_params = sum(dims[l + 1] * dims[l] + dims[l + 1] for l in range(len(acts)))
        self.row_stride = (off + 31) & ~31

    @staticmethod
    def from_module(model, n_actions, n_features):
        """Introspects Linear / ReLU / Tanh / Unflatten (utils/torch.py:19-22); anything else is rejected (no fallback)."""
        dims, acts, linears = [], [], []
        for m in model.children() if isinstance(model, torch.nn.Sequential) else [model]:
            if isinstance(m, torch.nn.Linear):
                if m.bias is None:
                    raise ValueError('psi Linear layers must have a bias')
                if not dims:
                    dims.append(m.in_features)
                elif m.in_features != dims[-1]:
                    raise ValueError('inconsistent layer widths in psi model')
                dims.append(m.out_features)
                acts.append('none')
                linears.append(m)
            elif isinstance(m, torch.nn.ReLU):
                acts[-1] = 'relu'
            elif isinstance(m, torch.nn.Tanh):
                acts[-1] = 'tanh'
            elif isinstance(m, (torch.nn.Unflatten, torch.nn.Identity)):
                pass
            else:
                raise TypeError(f'unsupported layer in psi model: {type(m).__name__} (Linear/ReLU/Tanh/Unflatten only)')
        return NetSpec(dims, acts, n_actions, n_features), linears

    def same_shape(self, other):
        return self.dims == other.dims and self.acts == other.acts

    def desc(self):
        d = _lib.NetDesc()
        d.n_layers = len(self.acts)
        for i, v in enumerate(self.dims):
            d.dims[i] = v
        for l in range(len(self.acts)):
            d.acts[l] = ACT[self.acts[l]]
            d.w_off[l] = self.w_off[l]
            d.b_off[l] = self.b_off[l]
        d.row_stride, d.n_actions, d.n_features = self.row_stride, self.n_actions, self.n_features
        return d

    def views(self, row):
        """[(W_l view, b_l view)] into one policy row."""
        out = []
        for l in range(len(self.acts)):
            o, i = self.dims[l + 1], self.dims[l]
            out.append((row[self.w_off[l]:self.w_off[l] + o * i].view(o, i), row[self.b_off[l]:self.b_off[l] + o]))
        return out


def _peer_flag_bytes():
    from .peer import FLAG_BYTES
    return FLAG_BYTES


def _peer_mode_ok(peer_mod):
    return peer_mod.peer_mode_wanted()


_raw_stream = getattr(torch._C, '_cuda_getCurrentRawStream', None)


def _stream():
    """torch's CURRENT stream on the current device as a raw handle (the fast getter when this torch has it: ~0.3 us vs ~5 us)."""
    if _raw_stream is not None:
        return C.c_void_p(_raw_stream(torch.cuda.current_device()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class _PsiFunction(torch.autograd.Function):
    """psi_j(x), j in [lo, lo+n_pol), as a function of the packed ONLINE rows and, on a library built with state_grad=True, of
    the states x (PackedSFLibrary.psi)."""

    @staticmethod
    def forward(ctx, online, lib, x, lo, n_pol):
        out, acts, masks = lib._psi_forward(x, lo, n_pol)
        # saved through save_for_backward: freed by the backward (unless retain_graph), a second backward raises
        ctx.save_for_backward(x, acts, masks)
        ctx.lib, ctx.lo, ctx.n_pol, ctx.gen, ctx.precision = lib, lo, n_pol, lib.weights_gen, lib.precision
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, d_psi):
        lib = ctx.lib
        if lib.weights_gen != ctx.gen:
            raise RuntimeError('one of the variables needed for gradient computation has been modified by an inplace operation: '
                               'the library\'s online psi rows were written (train step, optimizer step, add_policy or reset) '
                               'after this psi forward')
        if lib.precision != ctx.precision:       # the saved activations have the layout of the forward's mode
            raise RuntimeError(f'the library\'s precision mode changed from {ctx.precision!r} to {lib.precision!r} between this psi '
                               'forward and its backward')
        x, acts, masks = ctx.saved_tensors
        grad, dx = lib._psi_backward(x, ctx.lo, ctx.n_pol, acts, masks, d_psi, want_dx=ctx.needs_input_grad[2])
        return grad, None, dx, None, None


class PackedSFLibrary:
    def __init__(self, device=None, lr=None, wd=None, tsf_dim=None, capacity=4, precision='fp32', autograd=False,
                 state_grad=False):
        if state_grad and not autograd:
            raise ValueError('state_grad=True needs autograd=True')
        if not torch.cuda.is_available():
            raise RuntimeError('deep_successor_features_for_transfer_b200 needs a CUDA device (sm_100a); there is no CPU path')
        _lib.lib()                                   # fail loudly right here if the native library is missing
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        self.lr = dict(sf=1e-3, w=1e-3, g=1e-3, h=1e-3) if lr is None else dict(lr)
        self.wd = dict(sf=0.0, w=0.0, g=0.0, h=0.0) if wd is None else dict(wd)
        self.G = tsf_dim
        self.n_flows = 0            # planar flows ahead of g's Linear (normalising-flow g, tsfdqn_nf.py); set by the first add_policy
        self.spec = None
        self.n = 0
        self.cap = 0
        self._cap0 = capacity
        self._views = []            # per policy: dict of modules whose .data must be re-pointed after a re-pack
        self._ws = {}
        self.h = None
        self.shard = None           # dist.ShardContext once enable_sharding() was called
        self._xchg = None
        self._peer = None           # peer-memory exchange state (enable_sharding on an NVLink node)
        # autograd: the online storage is a leaf that requires grad, psi() records a differentiable forward and the packed
        # gradient [cap][row_stride] accumulates in online.grad.  weights_gen counts library-side writes of the online rows.
        self.autograd = bool(autograd)
        # state_grad: psi() also takes states that require grad and its backward returns dL/dx (sfgpi_mlp_input_grad)
        self.state_grad = bool(state_grad)
        self.weights_gen = 0
        self._grad_rows = set()     # rows whose gradient psi() backward has written since their optimizer's zero_grad
        self._bound_rows = set()    # ... of which the psi Linear modules' .grad are bound to their view of online.grad
        self.set_precision(precision)

    def set_precision(self, precision):
        """
        'fp32': CUDA-core FFMA kernels, 1e-5 parity with the reference.
        'bf16': every psi GEMM of the step -- the three forwards (online, GPI, target) AND the backward pass (dgrad chain,
        split-K wgrad) -- runs on the tcgen05 tensor cores with bf16 operands (states, weights, stored activations, dZ) and
        fp32 accumulation in TMEM; master weights, TD target / losses, g / h gradients and Adam stay fp32.  Stated tolerance:
        2e-2 scale-relative on psi / q, losses 3e-2, K-step weight / moment bounds in tests/test_gpu_bf16.py.
        'tf32x3': the same GEMMs on the tensor cores at the REFERENCE's precision -- tcgen05 kind::tf32 on fp32 operands split
        into hi + lo, three passes a_hi.b_hi + a_hi.b_lo + a_lo.b_hi, fp32 accumulation (csrc/mlp_stream_tc.cu): passes the
        fp32 mode's 1e-5 parity suite.  'tf32': one pass (operands rounded to tf32), stated tolerance 2e-3.
        """
        if precision not in ('fp32', 'bf16', 'tf32', 'tf32x3'):
            raise ValueError("precision must be 'fp32', 'bf16', 'tf32' or 'tf32x3'")
        self.precision = precision
        self._prec = _lib.PREC[precision]
        self._stream = precision in ('tf32', 'tf32x3')       # kind::tf32 streaming kernels on fp32 hi (/ lo) operand shadows
        self._parts = 2 if precision == 'tf32x3' else 1
        self._ws = {}
        self._shadow = {}

    def _shadow_for(self, which):
        """Operand shadow of the online / target rows, (re)allocated with the storage: bf16 [cap][rows][256], or for the tf32
        modes fp32 [parts][cap][rows][256] (hi, lo)."""
        buf = self._shadow.get(which)
        if buf is None or buf[1] != self.cap:
            desc = self.spec.desc()
            rpp = _lib.lib().sfgpi_bf16_rows_per_policy(C.byref(desc))
            if self._stream:
                buf = (torch.zeros(self._parts * self.cap * rpp * 256, dtype=torch.float32, device=self.device), self.cap)
            else:
                buf = (torch.zeros(self.cap * rpp * 256, dtype=torch.bfloat16, device=self.device), self.cap)
            self._shadow[which] = buf
        return buf[0]

    def _shadow_t(self):
        """tf32 modes: transposed operand shadows of the ONLINE rows for the dgrad chain: (W_l^T [parts][cap][L-2][256][256],
        W_out^T [parts][cap][256][ADp])."""
        buf = self._shadow.get('online_t')
        if buf is None or buf[2] != self.cap:
            desc = self.spec.desc()
            adp = _lib.lib().sfgpi_f32_out_pad(C.byref(desc))
            Lh = len(self.spec.acts) - 2
            buf = (torch.zeros(self._parts * self.cap * Lh * 256 * 256, dtype=torch.float32, device=self.device),
                   torch.zeros(self._parts * self.cap * 256 * adp, dtype=torch.float32, device=self.device), self.cap)
            self._shadow['online_t'] = buf
        return buf[0], buf[1]

    def _pack(self, which, lo, n_pol, transposed=False):
        desc = self.spec.desc()
        src = self.target if which == 'target' else self.online
        if self._stream:
            st, wt = self._shadow_t() if transposed else (None, None)
            _lib.call('sfgpi_pack_f32', C.byref(desc), ptr(src), lo, n_pol, self.cap, self._prec, ptr(self._shadow_for(which)),
                      ptr(st), ptr(wt), _stream())
        else:
            _lib.call('sfgpi_pack_bf16', C.byref(desc), ptr(src), lo, n_pol, ptr(self._shadow_for(which)), _stream())

    def _fold(self, a, which):
        """GPI form of the tensor-core forward: fold the reward vectors of `a` into the output layer -> (wq, bq)."""
        desc = self.spec.desc()
        nw = 1 if a.w_diag else a.n_w
        nq = _lib.lib().sfgpi_gpi_fold_rows(C.byref(desc), nw)
        key = ('fold', a.n_pol, nq)
        buf = self._ws.get(key)
        if buf is None:
            wq = torch.empty(self._parts * a.n_pol * nq * 256, dtype=torch.float32, device=self.device) if self._stream else \
                torch.empty(a.n_pol * nq * 256, dtype=torch.bfloat16, device=self.device)
            buf = self._ws[key] = (wq, self._f(a.n_pol * nq))
        wq, bq = buf
        src = self.target if which == 'target' else self.online
        if self._stream:
            _lib.call('sfgpi_fold_gpi_f32', C.byref(desc), ptr(src), a.policy_lo, a.n_pol, a.w, a.n_w, a.w_diag, self._prec, ptr(wq),
                      ptr(bq), _stream())
        else:
            _lib.call('sfgpi_fold_gpi', C.byref(desc), ptr(src), a.policy_lo, a.n_pol, a.w, a.n_w, a.w_diag, ptr(wq), ptr(bq), _stream())
        return wq, bq

    def _forward(self, a, which, fresh=False):
        """Dispatch one fused forward: fp32 CUDA-core kernel, or a tensor-core kernel on the operand shadow (packed on demand)."""
        if self.precision == 'fp32':
            _lib.call('sfgpi_mlp_forward', C.byref(a), _stream())
            return
        if not fresh:
            self._pack(which, a.policy_lo, a.n_pol)
        wq, bq = self._fold(a, which) if a.w else (None, None)     # GPI form
        if self._stream:
            job = _lib.ForwardTcJob()
            job.args, job.params_bf16, job.n_policies_total = a, self._shadow_for(which).data_ptr(), self.cap
            job.wq, job.bq = (wq.data_ptr(), bq.data_ptr()) if wq is not None else (None, None)
            _lib.call('sfgpi_mlp_forward_stream', C.byref(job), 1, self._prec, _stream())
        else:
            _lib.call('sfgpi_mlp_forward_tc', C.byref(a), ptr(self._shadow_for(which)), self.cap, ptr(wq), ptr(bq), _stream())

    def _forward_jobs(self, jobs, n):
        """Tensor-core mode: several forwards in ONE launch (jobs: ctypes array of ForwardTcJob, already filled in)."""
        _lib.call('sfgpi_mlp_forward_tc_jobs', C.byref(jobs), n, _stream())

    def enable_sharding(self, group=None):
        """Declare this library one policy shard of a multi-GPU ensemble (call on every rank after the tasks were added)."""
        from .dist import ShardContext
        self.shard = ShardContext(self.n, group)
        self._drop_plans()
        self._xchg = None
        if getattr(self, '_peer', None) is not None:         # re-sharding: no peer may still be pulling from the old arenas
            import torch.distributed as dist
            torch.cuda.synchronize(self.device)
            dist.barrier(group)
        self._close_peer()
        if self.shard.world > 1:
            D, sh = self.spec.n_features, self.shard
            nh = self.h.numel() if self.h is not None else 0
            x = dict(w_all=self._f(sh.n_total, D), nh=nh, ok=False)
            if sh.uniform:                                   # fused exchange: one all-gather per step (see _exchange)
                x.update(local=self._f(self.n * D + nh), all=self._f(sh.world, self.n * D + nh),
                         h_prev=self.h.clone() if nh else None)
            self._xchg = x
            import torch.distributed as dist
            from . import peer as _peer
            if sh.uniform and sh.world <= _lib.MAX_PEERS and dist.get_backend(group) == 'nccl' and _peer_mode_ok(_peer):
                # peer-memory exchange (csrc/peer.cu): flag block + double-buffered x_local in an arena every rank maps
                xb = (4 * (self.n * D + nh) + 15) // 16 * 16
                try:
                    arena = _peer.PeerArena(_peer.FLAG_BYTES + 2 * xb, group)
                    self._peer = dict(base=arena, xb=xb, ep=[0, 0], keys={})
                except RuntimeError as e:
                    import warnings
                    warnings.warn(f'peer-memory exchange unavailable, using NCCL collectives: {e}')
        return self.shard

    @property
    def _sharded(self):
        return self.shard is not None and self.shard.world > 1

    # ------------------------------------------------------------------ storage
    def _alloc(self, cap):
        sp, dev = self.spec, self.device
        z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)
        new = dict(online=z(cap, sp.row_stride), target=z(cap, sp.row_stride), m=z(cap, sp.row_stride),
                   v=z(cap, sp.row_stride), w=z(cap, sp.n_features), w_m=z(cap, sp.n_features), w_v=z(cap, sp.n_features),
                   step=torch.zeros(cap, dtype=torch.int32, device=dev),
                   # Adam bias corrections of every optimizer's NEXT step (t = step + 1), double like torch's host math
                   adam_consts=torch.tensor([[1.0 - 0.9 ** 1, math.sqrt(1.0 - 0.999 ** 1)]], dtype=torch.float64,
                                            device=dev).repeat(cap, 1).contiguous(),
                   # ... and its twin: the train step's Adam launch reads one buffer and writes the next step's corrections
                   # into the other (sfgpi_adam_args.consts_next); _adam_par[i] says which buffer is current for policy i
                   adam_consts2=torch.tensor([[1.0 - 0.9 ** 1, math.sqrt(1.0 - 0.999 ** 1)]], dtype=torch.float64,
                                             device=dev).repeat(cap, 1).contiguous())
        if self.G is not None:
            gl = self.G * sp.dims[0] + self.G + self.n_flows * (2 * sp.dims[0] + 1)      # W | b | K x (weight | bias | scale)
            hl = sp.n_features * self.G + sp.n_features
            new.update(g=z(cap, gl), g_m=z(cap, gl), g_v=z(cap, gl), h_m=z(cap, hl), h_v=z(cap, hl))
        old_grad = getattr(self, 'online', None)
        old_grad = None if old_grad is None else old_grad.grad
        with torch.no_grad():
            for k, t in new.items():
                old = getattr(self, k, None)
                if old is not None and self.n > 0:
                    t[:self.n].copy_(old[:self.n])
                setattr(self, k, t)
        if self.autograd:
            self.online.requires_grad_(True)
            self.online.register_post_accumulate_grad_hook(PackedSFLibrary._grad_hook(self))
            if old_grad is not None:
                self.online.grad = torch.zeros_like(self.online)
                self.online.grad[:self.n].copy_(old_grad[:self.n])
            self._bound_rows = set()
        self.cap = cap
        self._adam_par = (getattr(self, '_adam_par', None) or []) + [0] * (cap - len(getattr(self, '_adam_par', None) or []))
        self._ws = {}
        self.invalidate_exchange()
        for i, mods in enumerate(self._views):
            self._point_views(i, mods)
        if self.autograd:
            self._bind_grads()

    def _point_views(self, i, mods):
        for (W, b), lin in zip(self.spec.views(self.online.detach()[i]), mods['online']):
            lin.weight.data, lin.bias.data = W, b
            if self.autograd:                                # (re)bound to online.grad by _bind_grads
                lin.weight.grad = lin.bias.grad = None
        for (W, b), lin in zip(self.spec.views(self.target[i]), mods['target']):
            lin.weight.data, lin.bias.data = W, b
        mods['w'].weight.data = self.w[i].view(1, -1)
        if mods.get('g') is not None:
            S = self.spec.dims[0]
            flows, lin = self._split_g(mods['g'])
            lin.weight.data = self.g[i, :self.G * S].view(self.G, S)
            lin.bias.data = self.g[i, self.G * S:self.G * S + self.G]
            for k, f in enumerate(flows):
                o = self.G * S + self.G + k * (2 * S + 1)
                f.weight.data, f.bias.data, f.scale.data = self.g[i, o:o + S].view(1, S), self.g[i, o + S:o + S + 1], self.g[i, o + S + 1:o + 2 * S + 1].view(1, S)

    @staticmethod
    def _split_g(g):
        """g-function module -> (planar flows, final Linear): nn.Linear (tsfdqn.py:537-539) or Sequential(flows..., Linear) (tsfdqn_nf.py:352-358)."""
        if isinstance(g, torch.nn.Linear):
            return [], g
        mods = list(g)
        return mods[:-1], mods[-1]

    def add_policy(self, model, target_model, w_linear, g_linear=None, h_linear=None, n_actions=None, n_features=None):
        """Adopts freshly built reference-style modules into packed storage (sfdqn.py:180-288)."""
        spec, lin_on = NetSpec.from_module(model, n_actions, n_features)
        spec_t, lin_tg = NetSpec.from_module(target_model, n_actions, n_features)
        if self.spec is None:
            self.spec = spec
        if not (self.spec.same_shape(spec) and self.spec.same_shape(spec_t)):
            raise ValueError('all psi networks of a library must share one architecture')
        if (g_linear is None) != (self.G is None):
            raise ValueError('g/h functions must be given iff the library was built with tsf_dim')
        if g_linear is not None:
            flows, g_lin = self._split_g(g_linear)
            if self.n == 0 and self.n_flows != len(flows):
                self.n_flows, self.cap = len(flows), 0           # (re-allocated below with the g row's real length)
            if len(flows) != self.n_flows:
                raise ValueError('every g function of a library must have the same number of flows')
        if self.n == self.cap:
            self._alloc(max(self._cap0, 2 * self.cap))
        i = self.n
        with torch.no_grad():
            for (W, b), lin in zip(self.spec.views(self.online[i]), lin_on):
                W.copy_(lin.weight.data)
                b.copy_(lin.bias.data)
            for (W, b), lin in zip(self.spec.views(self.target[i]), lin_tg):
                W.copy_(lin.weight.data)
                b.copy_(lin.bias.data)
            self.w[i].copy_(w_linear.weight.data.reshape(-1))
            mods = dict(online=lin_on, target=lin_tg, w=w_linear, g=g_linear)
            if g_linear is not None:
                S = self.spec.dims[0]
                if g_lin.out_features != self.G or g_lin.in_features != S:
                    raise ValueError('g function shape mismatch')
                self.g[i, :self.G * S].copy_(g_lin.weight.data.reshape(-1))
                self.g[i, self.G * S:self.G * S + self.G].copy_(g_lin.bias.data)
                for k, f in enumerate(flows):
                    o = self.G * S + self.G + k * (2 * S + 1)
                    self.g[i, o:o + 2 * S + 1].copy_(torch.cat([f.weight.data.reshape(-1), f.bias.data.reshape(-1), f.scale.data.reshape(-1)]))
                if self.h is None:
                    D = self.spec.n_features
                    self.h = torch.cat([h_linear.weight.data.reshape(-1), h_linear.bias.data.reshape(-1)]).float().to(self.device).contiguous()
                    h_linear.weight.data = self.h[:D * self.G].view(D, self.G)
                    h_linear.bias.data = self.h[D * self.G:]
                    self.h_module = h_linear
        self._views.append(mods)
        self._point_views(i, mods)
        self.n += 1
        self.weights_gen += 1
        # cached train-step plans hard-code the policy count (GPI range, pack range, 'all' = n policies): drop them
        self._drop_plans()
        self.invalidate_exchange()
        return i

    def _drop_plans(self):
        self._ws = {k: v for k, v in self._ws.items() if not (isinstance(k, tuple) and k and k[0] == 'plan')}

    def _close_peer(self):
        """Unmap / free the peer arenas (collective-free: every rank just releases its own mappings and allocation)."""
        pa, self._peer = getattr(self, '_peer', None), None
        if pa is not None:
            torch.cuda.synchronize(self.device)              # no kernel of this rank may still touch a mapping
            for arena in [pa['base']] + list(pa['keys'].values()):
                arena.close()

    def __del__(self):
        try:
            self._close_peer()
        except Exception:
            pass

    def reset(self):
        self._close_peer()
        self.spec, self.n, self.cap, self._views, self._ws, self.h = None, 0, 0, [], {}, None
        self._adam_par = []
        self.weights_gen += 1
        self._grad_rows, self._bound_rows = set(), set()
        for k in ('online', 'target', 'm', 'v', 'w', 'w_m', 'w_v', 'step', 'adam_consts', 'adam_consts2', 'g', 'g_m', 'g_v', 'h_m', 'h_v'):
            if hasattr(self, k):
                delattr(self, k)

    # ------------------------------------------------------------------ workspaces
    def _f(self, *shape):
        return torch.empty(*shape, dtype=torch.float32, device=self.device)

    def _hidden_storage(self, n_pol, B, new, precision=None):
        """
        Storage for hidden layers 0..L-2 of n_pol nets at batch B in mode `precision` (default: the library's) -> (values,
        ReLU mask words).  Saved activations and dZ have these shapes in every mode.
          fp32:          one flat fp32 buffer holding every layer's [n_pol][B][dims[l+1]] (views: _fp32_acts); masks None
          bf16:          bf16 [L-1][n_pol][B][256]
          tf32 / tf32x3: fp32 [parts][L-1][n_pol][B][256] (hi (, lo)), row-major, written by TMA and read back MN-major by wgrad
        The tensor-core modes' masks are int32 [L-1][n_pol][B][8].  new: torch.empty or torch.zeros.
        """
        sp, L, dev = self.spec, len(self.spec.acts), self.device
        precision = precision or self.precision
        if precision == 'fp32':
            return new(n_pol * B * sum(sp.dims[1:L]), dtype=torch.float32, device=dev), None
        if precision == 'bf16':
            values = new(L - 1, n_pol, B, 256, dtype=torch.bfloat16, device=dev)
        else:
            values = new(2 if precision == 'tf32x3' else 1, L - 1, n_pol, B, 256, dtype=torch.float32, device=dev)
        return values, new(L - 1, n_pol, B, 8, dtype=torch.int32, device=dev)

    def _fp32_scratch(self, n_pol, B):
        """Scratch of the fp32 backward kernels for n_pol nets at batch B, whatever the library's mode (the G4 step runs them
        in every mode): saved activations, dZ, the split-K count and the weight-gradient partials [n_pol][n_split][row_stride]."""
        sp, L = self.spec, len(self.spec.acts)
        acts, masks = self._hidden_storage(n_pol, B, torch.zeros, 'fp32')
        tiles = sum(((sp.dims[l + 1] + 63) // 64) * ((sp.dims[l] + 255) // 256) for l in range(L))
        n_split = max(1, min((B + 127) // 128, -(-296 // (tiles * n_pol))))
        return dict(acts=acts, masks=masks, dz=torch.zeros_like(acts), n_split=n_split,
                    grad_part=torch.zeros(n_pol, n_split, sp.row_stride, dtype=torch.float32, device=self.device))

    def _workspace(self, B, n_pol):
        """Scratch of the train step, psi_gradients and the psi() backward for n_pol nets at batch B: the backward's (acts,
        masks, dz, in the tensor-core modes dzo / xo, grad_part, n_split) and the TD step's buffers."""
        key = (B, n_pol)
        ws = self._ws.get(key)
        if ws is None:
            sp = self.spec
            L, D = len(sp.acts), sp.n_features
            if self.precision == 'fp32':
                ws = self._fp32_scratch(n_pol, B)
            else:
                # tensor-core backward: row-major activations / dZ (MN-major UMMA operands), split-K over the batch in one
                # wave of CTAs
                acts, masks = self._hidden_storage(n_pol, B, torch.zeros)
                lib, desc = _lib.lib(), sp.desc()
                adp = (lib.sfgpi_f32_out_pad if self._stream else lib.sfgpi_bwd_tc_out_pad)(C.byref(desc))
                lead = (self._parts,) if self._stream else ()
                items = (sp.dims[-1] + 127) // 128 + 2 * (L - 1)
                n_split = lib.sfgpi_bwd_tc_splits(B, max(1, 148 // (items * n_pol)))
                ws = dict(acts=acts, masks=masks, dz=torch.zeros_like(acts), dzo=acts.new_zeros(*lead, n_pol, B, adp),
                          xo=acts.new_zeros(*lead, B, 32 if self._stream else 64), n_split=n_split,
                          grad_part=torch.zeros(n_pol, n_split, sp.row_stride, dtype=torch.float32, device=self.device))
            ws.update(cur_sel=self._f(n_pol, B, D), next_sel=self._f(n_pol, B, D), d_out=self._f(n_pol, B, D),
                      keys=torch.empty(n_pol, B, dtype=torch.int64, device=self.device))
            nblk = _lib.lib().sfgpi_td_partials(B)        # one TD partial per 8-CTA cluster (256 transitions)
            ws['nblk'] = nblk
            ws['loss_part'] = self._f(n_pol, nblk, 2)
            if self.G is not None:
                S = sp.dims[0]
                ws['aux_len'] = D + self.g.shape[1] + D * self.G + D
            else:
                ws['aux_len'] = D
            ws['aux_part'] = self._f(n_pol, nblk, ws['aux_len'])
            if self.G is not None:
                ws['tsf_part'] = self._f(n_pol, nblk, 2 * D + D * sp.dims[0] + self.n_flows * (2 * sp.dims[0] + 1))
            self._ws[key] = ws
        return ws

    # ------------------------------------------------------------------ forward-only entry points
    def _check_x(self, x):
        x = torch.as_tensor(x)
        if x.dim() == 1:
            x = x.unsqueeze(0)
        x = x.to(device=self.device, dtype=torch.float32).contiguous()
        if x.dim() != 2 or x.shape[1] != self.spec.dims[0]:
            raise ValueError(f'expected states of shape [B, {self.spec.dims[0]}], got {tuple(x.shape)}')
        return x

    def _fwd_args(self, params, lo, n_pol, x, B=None):
        a = _lib.ForwardArgs()
        a.net = self.spec.desc()
        a.params, a.policy_lo, a.n_pol = ptr(params), lo, n_pol
        a.x, a.B = ptr(x), (x.shape[0] if B is None else B)
        a.mode = 0
        return a

    def forward_psi(self, x, lo=0, n_pol=None, target=False):
        """psi_j(x) for j in [lo, lo+n_pol): [B][n_pol][A][D] (get_successors / get_next_successors)."""
        if target and self.state_grad and torch.is_grad_enabled() and isinstance(x, torch.Tensor) and x.requires_grad:
            # a result without a backward would silently cut the states' gradient; torch would raise or differentiate
            raise RuntimeError('the target psi nets are constants and have no gradient with respect to the states: call them under '
                               'torch.no_grad() or pass the states .detach()ed')
        x = self._check_x(x)
        n_pol = self.n - lo if n_pol is None else n_pol
        sp = self.spec
        out = self._f(x.shape[0], n_pol, sp.n_actions, sp.n_features)
        a = self._fwd_args(self.target if target else self.online, lo, n_pol, x)
        a.psi_out = ptr(out)
        self._forward(a, 'target' if target else 'online')
        return out

    def psi(self, x, lo=0, n_pol=None):
        """
        Differentiable psi_j(x), j in [lo, lo+n_pol) of the ONLINE nets: [B][n_pol][A][D], equal to forward_psi bit for bit.
        Under grad mode the result carries a backward that runs the precision mode's backward kernels on the dense dL/dpsi and
        accumulates dL/d(row) into online.grad ([cap][row_stride], library row layout); every psi Linear of a row that received
        a gradient then has its .grad bound to its view of that buffer.  Needs a library built with autograd=True.  The
        backward raises if the library wrote the online rows after this forward (weights_gen).
        States that require grad are refused unless the library was built with state_grad=True.  Then the backward also returns
        dL/dx = sum_j dZ0_j . W0_j over the n_pol nets (one sfgpi_mlp_input_grad launch on the layer-0 gradient the backward
        kernels leave in their scratch), and autograd carries it back through the dtype / device conversion and the
        unsqueeze of a 1-D state, so x.grad has x's own dtype and shape.  States that do not require grad cost nothing extra.
        """
        if not self.autograd:
            raise RuntimeError('psi() needs a library built with autograd=True')
        if self._sharded:
            raise NotImplementedError('psi() does not support sharded libraries')
        if isinstance(x, torch.Tensor) and x.requires_grad:
            if not self.state_grad:
                raise ValueError('psi() has no gradient with respect to the states: pass x.detach(), or build the library with '
                                 'state_grad=True')
            if self.spec is not None and len(self.spec.acts) < 2:
                raise NotImplementedError('state gradients need a psi net with at least one hidden layer')
        x = self._check_x(x)
        n_pol = self.n - lo if n_pol is None else n_pol
        if not (0 <= lo and n_pol >= 1 and lo + n_pol <= self.n):
            raise IndexError('policy range out of bounds')
        return _PsiFunction.apply(self.online, self, x, lo, n_pol)

    def _psi_forward(self, x, lo, n_pol):
        """forward_psi that also keeps what the backward needs: activations (and ReLU masks) allocated for this call alone,
        because several recorded forwards (e.g. psi(s) and psi(s')) can be alive at once.  Returns (psi, acts, masks): fp32
        mode, acts is one flat buffer holding every hidden layer's [n_pol][B][width] (see _fp32_acts) and masks is None.
        torch.empty: the forward kernels store every activation the backward reads (every row < B, all 256 columns of the
        tensor-core layouts, the mask words of every ReLU layer; masks of other layers are never read)."""
        sp, B = self.spec, x.shape[0]
        out = self._f(B, n_pol, sp.n_actions, sp.n_features)
        a = self._fwd_args(self.online, lo, n_pol, x)
        a.psi_out = ptr(out)
        acts, masks = self._hidden_storage(n_pol, B, torch.empty)
        self._save_acts(a, acts, masks)
        self._forward(a, 'online')
        return out, acts, masks

    def _fp32_acts(self, flat, n_pol, B):
        """Per-layer [n_pol][B][dims[l+1]] views of the fp32 mode's flat activation buffer."""
        sp, out, off = self.spec, [], 0
        for l in range(len(sp.acts) - 1):
            n = n_pol * B * sp.dims[l + 1]
            out.append(flat[off:off + n].view(n_pol, B, sp.dims[l + 1]))
            off += n
        return out

    def _save_acts(self, a, acts, masks):
        """Point forward args `a` at the storage (_hidden_storage) for the activations it saves: per-layer fp32 views when
        masks is None, else the tensor-core layout and its ReLU mask words."""
        if masks is None:
            for l, t in enumerate(self._fp32_acts(acts, a.n_pol, a.B)):
                a.acts_out[l] = t.data_ptr()
        else:
            a.acts_bf16_out, a.relu_mask_out = acts.data_ptr(), masks.data_ptr()

    def _fp32_backward(self, scratch, lo, n_pol, B, acts=None):
        """BackwardArgs of the fp32 kernels over `scratch` (_fp32_scratch) for this library's nets [lo, lo+n_pol), whatever
        its mode; acts: saved activations outside the scratch."""
        b = _lib.BackwardArgs()
        b.net, b.params, b.policy_lo, b.n_pol, b.B = self.spec.desc(), ptr(self.online), lo, n_pol, B
        acts = self._fp32_acts(scratch['acts'] if acts is None else acts, n_pol, B)
        for l, (h, dz) in enumerate(zip(acts, self._fp32_acts(scratch['dz'], n_pol, B))):
            b.acts[l], b.dz[l] = h.data_ptr(), dz.data_ptr()
        b.grad_part, b.n_split = ptr(scratch['grad_part']), scratch['n_split']
        return b

    def _backward_args(self, ws, lo, n_pol, B, acts=None, masks=None):
        """
        The mode's backward argument block for nets [lo, lo+n_pol) at batch B over workspace `ws` -> (args, C entry point,
        sfgpi_run op).  acts / masks: the saved activations of a forward outside the workspace (psi()), else ws's.  The caller
        sets x, actions (NULL: d_out is a dense dL/dpsi) and d_out; the train step also xo_ready / expand_td.
        """
        if self.precision == 'fp32':
            return self._fp32_backward(ws, lo, n_pol, B, acts), 'sfgpi_mlp_backward', 'BACKWARD'
        if acts is None:
            acts, masks = ws['acts'], ws['masks']
        if self._stream:
            b = _lib.BackwardStreamArgs()
            sh_t, wo_t = self._shadow_t()
            b.precision, b.shadow_t, b.wout_t = self._prec, ptr(sh_t), ptr(wo_t)
            b.acts, b.dz, b.dzo, b.xo = ptr(acts), ptr(ws['dz']), ptr(ws['dzo']), ptr(ws['xo'])
            entry, op = 'sfgpi_mlp_backward_stream', 'BACKWARD_STREAM'
        else:
            b = _lib.BackwardTcArgs()
            b.params_bf16 = ptr(self._shadow_for('online'))
            b.acts_bf16, b.dz_bf16, b.dzo_bf16, b.xo_bf16 = ptr(acts), ptr(ws['dz']), ptr(ws['dzo']), ptr(ws['xo'])
            entry, op = 'sfgpi_mlp_backward_tc', 'BACKWARD_TC'
        b.net, b.n_policies_total, b.relu_masks = self.spec.desc(), self.cap, ptr(masks)
        b.policy_lo, b.n_pol, b.B = lo, n_pol, B
        b.grad_part, b.n_split = ptr(ws['grad_part']), ws['n_split']
        return b, entry, op

    def _psi_backward(self, x, lo, n_pol, acts, masks, d_psi, want_dx=False):
        """Dense-d_out backward of one psi() forward -> (gradient w.r.t. the whole online storage (rows outside zero), dL/dx
        [B][S] when want_dx, else None)."""
        B = x.shape[0]
        d_psi = d_psi.to(torch.float32).contiguous()                 # [B][n_pol][A][D]: the psi_out layout the kernels read
        ws = self._workspace(B, n_pol)
        if self.precision != 'fp32':                      # the backward's operands (tf32: transposed)
            self._pack('online', lo, n_pol, transposed=True)
        b, entry, _ = self._backward_args(ws, lo, n_pol, B, acts, masks)
        b.x, b.actions, b.d_out = x.data_ptr(), None, d_psi.data_ptr()          # actions NULL: d_out is dense
        _lib.call(entry, C.byref(b), _stream())
        dx = self._input_grad(ws, lo, n_pol, B) if want_dx else None     # while dZ_0 is in the workspace
        if self.online.grad is not None:
            # rows whose psi .grad a stock torch optimizer's zero_grad() set to None: start their accumulation afresh
            for i in sorted(self._bound_rows & set(range(lo, lo + n_pol))):
                if all(p.grad is None for lin in self._views[i]['online'] for p in (lin.weight, lin.bias)):
                    self.online.grad[i].zero_()
                    self._bound_rows.discard(i)
        grad = torch.zeros(self.online.shape, dtype=torch.float32, device=self.device)
        torch.sum(ws['grad_part'], dim=1, out=grad[lo:lo + n_pol])
        self._grad_rows.update(range(lo, lo + n_pol))
        return grad, dx

    def _input_grad(self, ws, lo, n_pol, B):
        """dL/dx [B][S] = sum_j dZ0_j . W0_j from the layer-0 gradient the last backward into workspace `ws` left there."""
        g = ws.get('input_grad')
        if g is None:                                                # built once per workspace (dropped with the storage)
            g = ws['input_grad'] = _lib.InputGradArgs()
            g.net, g.precision, g.params, g.n_pol, g.B = self.spec.desc(), self._prec, ptr(self.online), n_pol, B
            g.dz0 = ptr(ws['dz'])                                    # layer 0 (of part 0) starts every mode's layout
            if self._stream:                                         # [parts][L-1][n_pol][B][256]: slab 0 of each part
                g.dz0_part_stride = ws['dz'][0].numel()
        dx = self._f(B, self.spec.dims[0])
        g.policy_lo, g.dx = lo, dx.data_ptr()
        _lib.call('sfgpi_mlp_input_grad', C.byref(g), _stream())
        return dx

    @staticmethod
    def _grad_hook(lib):
        """post-accumulate-grad hook of the online storage: bind the psi Linear .grad of every row with a gradient to its view
        of online.grad, so that stock torch code (clip_grad_norm_, torch.optim over sf.psi[i][0][0].parameters()) reads the
        packed gradient and its in-place changes reach it."""
        import weakref
        ref = weakref.ref(lib)

        def hook(online):
            self = ref()
            if self is not None:
                self._bind_grads()
        return hook

    def _bind_grads(self):
        if self.online.grad is None:
            return
        g = self.online.grad.detach()
        for i in sorted(self._grad_rows - self._bound_rows):
            for (W, b), lin in zip(self.spec.views(g[i]), self._views[i]['online']):
                lin.weight.grad, lin.bias.grad = W, b
            self._bound_rows.add(i)

    def gpi(self, x, w_vec, lo=0, n_pol=None, want_q=True, task_base=None, keys_out=None, reduce=True):
        """
        Fused GPI_w (sfdqn.py:215-240): returns (q [B][n_pol][A] or None, key_action [B], key_task [B]) -- packed int64
        keys, decode with decode_keys().  psi[B,N,A,D] is never materialised.
        """
        x = self._check_x(x)
        n_pol = self.n - lo if n_pol is None else n_pol
        B, sp = x.shape[0], self.spec
        w_vec = w_vec.detach().to(device=self.device, dtype=torch.float32).reshape(-1).contiguous()
        if w_vec.numel() != sp.n_features:
            raise ValueError('reward vector must have n_features elements')
        keys = torch.empty(2, B, dtype=torch.int64, device=self.device) if keys_out is None else keys_out
        _lib.call('sfgpi_keys_fill', ptr(keys), 2 * B, _stream())
        q = self._f(B, n_pol, sp.n_actions) if want_q else None
        a = self._fwd_args(self.online, lo, n_pol, x)
        a.w, a.n_w, a.w_diag = ptr(w_vec), 1, 0
        a.key_action, a.key_task = C.c_void_p(keys[0].data_ptr()), C.c_void_p(keys[1].data_ptr())
        a.task_base = (self.shard.lo + lo if self.shard is not None else lo) if task_base is None else task_base
        a.q_out = ptr(q)
        self._forward(a, 'online')
        if self._sharded and reduce:
            from .dist import allreduce_max_keys
            allreduce_max_keys(keys, self.shard.group)          # packed (value,index) MAX over NVLink: global GPI
        return q, keys[0], keys[1]

    def gpi_select(self, x, w_vec, lo=0, n_pol=None):
        """
        Caller-side selection of the agents (sfdqn.py:585-594, tsfdqn.py:529-535) straight from the packed keys the fused GPI
        kernel produces: returns an int64 device tensor [2][B], row 0 = argmax_a max_j q (the greedy action), row 1 =
        argmax_j max_a q (the policy active in GPI, global index) -- no q[B,N,A] tensor, no eager indexing / argmax launches.
        With (lo, n_pol) = (i, 1) row 0 is argmax_a q_i: the `use_gpi=False` selection, at the cost of ONE net instead of N.
        Tie clause: the reference takes the first maximal task and then the first maximal action of THAT task's row; the key
        takes the smallest action among all cells holding the maximum -- they differ only under exact fp32 ties across policies.
        The result lives in a per-batch-size workspace and is valid until the next gpi_select call of the same size.
        """
        x = self._check_x(x)
        n_pol = self.n - lo if n_pol is None else n_pol
        B = x.shape[0]
        ws = self._ws.get(('select', B))
        if ws is None:
            ws = self._ws[('select', B)] = (torch.empty(2, B, dtype=torch.int64, device=self.device),
                                            torch.empty(2, B, dtype=torch.int64, device=self.device))
        keys, idx = ws
        self.gpi(x, w_vec, lo, n_pol, want_q=False, keys_out=keys)
        _lib.call('sfgpi_keys_decode', ptr(keys), 2 * B, ptr(idx), None, _stream())
        return idx

    def decode_keys(self, keys, want_value=False):
        idx = torch.empty(keys.shape, dtype=torch.int64, device=self.device)
        val = self._f(*keys.shape) if want_value else None
        _lib.call('sfgpi_keys_decode', ptr(keys), keys.numel(), ptr(idx), ptr(val), _stream())
        return (idx, val) if want_value else idx

    def gpi_from_psi(self, psi, w_vec, task_base=0, want_q=True):
        """Unfused GPI epilogue on a materialised psi [B][N][A][D]."""
        psi = psi.to(device=self.device, dtype=torch.float32).contiguous()
        B, N, A, D = psi.shape
        w_vec = w_vec.detach().to(device=self.device, dtype=torch.float32).reshape(-1).contiguous()
        keys = torch.empty(2, B, dtype=torch.int64, device=self.device)
        q = self._f(B, N, A) if want_q else None
        _lib.call('sfgpi_gpi_from_psi', ptr(psi), ptr(w_vec), B, N, A, D, task_base, ptr(q),
                  C.c_void_p(keys[0].data_ptr()), C.c_void_p(keys[1].data_ptr()), _stream())
        return q, keys[0], keys[1]

    # ------------------------------------------------------------------ the train step
    def _build_plan(self, B, policy, use_gpi, variant, beta):
        """Pre-builds every C-ABI argument block of one train step; only the six input pointers change per call."""
        sp = self.spec
        D, A, S = sp.n_features, sp.n_actions, sp.dims[0]
        ensemble = policy == 'all'
        lo, n_pol = (0, self.n) if ensemble else (int(policy), 1)
        if not (0 <= lo < self.n):
            raise IndexError('policy index out of range')
        ws = self._workspace(B, n_pol)
        keys = ws['keys']
        P = lambda tns, i=lo: C.c_void_p(tns[i].data_ptr())

        # (1) online forward on s: saves hidden outputs, gathers psi(s)[a_b]            sfdqn.py:328
        a1 = self._fwd_args(self.online, lo, n_pol, None, B)
        tc = self.precision != 'fp32'
        st_mode = self._stream
        self._save_acts(a1, ws['acts'], ws['masks'])
        a1.sel_out = ptr(ws['cur_sel'])
        # (2) next actions: GPI over the whole library (or own psi) with w_i            sfdqn.py:314-322
        #     sharded: this rank scores its local policies for ALL n_total reward vectors (gathered into w_all); the
        #     per-rank keys [n_total][B] are MAX-all-reduced, then rows [shard.lo, shard.lo + n) are this rank's own.
        sharded = self._sharded and use_gpi
        if sharded and not ensemble:
            raise NotImplementedError('sharded libraries step all local policies at once (policy="all"); the single-policy '
                                      'step with cross-GPU GPI is train_step_owner()/gpi_assist()')
        key_row0 = 0
        w_all = None
        peer = None
        if use_gpi:
            a2 = self._fwd_args(self.online, 0, self.n, None, B)
            if sharded and ensemble:
                nt = self.shard.n_total
                w_all = self._xchg['w_all']
                a2.w, a2.n_w, a2.w_diag, key_row0 = ptr(w_all), nt, 0, self.shard.lo
                if getattr(self, '_peer', None) is not None and not st_mode:
                    # peer mode: this rank's keys [nt][B] live in a mapped arena (double-buffered on epoch parity); the
                    # exchange kernel leaves the MAX over ranks of this rank's own rows in keys_own
                    from .peer import PeerArena
                    kb = (nt * B * 8 + 15) // 16 * 16      # halves stay 16-byte aligned (128-bit peer loads)
                    karena = self._peer['keys'].get(B)
                    if karena is None:
                        karena = self._peer['keys'][B] = PeerArena(2 * kb, self.shard.group)
                    peer = dict(karena=karena, kb=kb, lo=self.shard.lo)
                    keys = ws['keys_own'] = ws.get('keys_own', torch.empty(n_pol, B, dtype=torch.int64, device=self.device))
                    key_row0 = 0
                else:
                    keys = ws['keys_all'] = ws.get('keys_all', torch.empty(nt, B, dtype=torch.int64, device=self.device))
            else:
                a2.w, a2.n_w, a2.w_diag = P(self.w), n_pol, 0
            a2.task_base = self.shard.lo if self.shard is not None else 0
        else:
            a2 = self._fwd_args(self.online, lo, n_pol, None, B)
            a2.w, a2.n_w, a2.w_diag = P(self.w), n_pol, 1
        a2.key_action = ptr(keys)
        # (3) target forward on s', gather psi^-(s')[a*]                                sfdqn.py:330-331
        a3 = self._fwd_args(self.target, lo, n_pol, None, B)
        if tc:
            # tensor-core mode: the three forwards share one launch, so the target nets cannot wait for a*; they emit the full
            # psi^-(s') [B][n_pol][A*D] and the TD kernel gathers row a* by the (all-reduced) GPI key.
            if 'next_psi' not in ws:
                ws['next_psi'] = self._f(B, n_pol, A * D)
            a3.psi_out = ptr(ws['next_psi'])
        else:
            a3.sel_keys, a3.sel_key_stride, a3.sel_out = C.c_void_p(keys[key_row0:].data_ptr()), B, ptr(ws['next_sel'])
        # (4) TD target, losses, d_out and the reward-head / g / h gradients            sfdqn.py:330-345, tsfdqn.py:621-645
        t = _lib.TdArgs()
        t.variant, t.n_pol, t.B, t.S, t.A, t.D, t.G = variant, n_pol, B, S, A, D, (self.G or 0)
        t.beta = float(beta) if variant == 2 else 1.0
        t.cur_sel, t.next_sel = ptr(ws['cur_sel']), ptr(ws['next_sel'])
        if tc:
            t.next_psi, t.next_keys, t.next_key_stride = ptr(ws['next_psi']), C.c_void_p(keys[key_row0:].data_ptr()), B
        t.w, t.w_stride = P(self.w), D
        if variant == 2:
            t.g, t.g_stride, t.h, t.n_flows = P(self.g), self.g.shape[1], ptr(self.h), self.n_flows
        t.d_out, t.loss_part, t.aux_grad_part, t.aux_len = ptr(ws['d_out']), ptr(ws['loss_part']), ptr(ws['aux_part']), ws['aux_len']
        if variant == 2:
            t.tsf_part = ptr(ws['tsf_part'])
        # (5) backward through psi: dgrad chain + split-K wgrad
        b, _, b_op = self._backward_args(ws, lo, n_pol, B)
        b.d_out = ptr(ws['d_out'])
        if variant == 2 and b_op == 'BACKWARD_TC':
            t.defer_expand, b.expand_td = 1, C.addressof(t)            # TSF expand rides in the dgrad launch (idle SMs)
        # (6) Adam over (psi | w | g | h) for all stepped optimizers, + loss reduction    sfdqn.py:362, tsfdqn.py:700
        ad = _lib.AdamArgs()
        ad.n_pol, ad.step = n_pol, C.c_void_p(self.step[lo:].data_ptr())
        ad.consts = C.c_void_p(self.adam_consts[lo:].data_ptr())          # (consts / consts_next: patched per step, see train_step)
        ad.beta1, ad.beta2, ad.eps = 0.9, 0.999, 1e-8
        rs_, nblk, al = sp.row_stride, ws['nblk'], ws['aux_len']
        npa = 1 if variant == 2 else nblk          # variant 2: the TD step leaves ONE reduced aux-gradient row per policy

        def seg(k, param, pstride, m, v, mstride, grad, gpol, gpart, npart, length, lr, wd):
            s = ad.seg[k]
            s.param, s.param_stride, s.m, s.m_stride, s.v, s.v_stride = param, pstride, m, mstride, v, mstride
            s.grad_part, s.grad_pol_stride, s.grad_part_stride, s.n_part = grad, gpol, gpart, npart
            s.len, s.lr, s.weight_decay = length, lr, wd

        seg(0, P(self.online), rs_, P(self.m), P(self.v), rs_, ptr(ws['grad_part']), ws['n_split'] * rs_, rs_, ws['n_split'],
            rs_, self.lr['sf'], self.wd['sf'])
        nseg = 1
        aux = ws['aux_part']
        if variant >= 1:
            seg(1, P(self.w), D, P(self.w_m), P(self.w_v), D, ptr(aux), nblk * al, al, npa, D, self.lr['w'], self.wd['w'])
            nseg = 2
        if variant == 2:
            gl, hl = self.g.shape[1], self.h.numel()
            seg(2, P(self.g), gl, P(self.g_m), P(self.g_v), gl, C.c_void_p(aux.data_ptr() + 4 * D), nblk * al, al, npa, gl,
                self.lr['g'], self.wd['g'])
            seg(3, ptr(self.h), 0, P(self.h_m), P(self.h_v), hl, C.c_void_p(aux.data_ptr() + 4 * (D + gl)), nblk * al, al, npa,
                hl, self.lr['h'], self.wd['h'])
            nseg = 4
        ad.n_seg = nseg
        ad.loss_part, ad.n_loss_part = ptr(ws['loss_part']), nblk
        ad.l1_scale, ad.l2_scale = 1.0 / (B * A * D), 1.0 / B
        ad.beta_loss = (float(beta) if variant == 2 else 1.0) if variant >= 1 else 0.0
        ad.sequential_shared = 1
        return dict(ws=ws, a1=a1, a2=a2, a3=a3, t=t, b=b, b_op=b_op, ad=ad, n_pol=n_pol, lo=lo, tc=tc, st=st_mode, B=B, ring=0, keys=keys, w_all=w_all, sharded=sharded,
                    peer=peer, variant=variant,
                    losses=torch.zeros(64, n_pol, 3, dtype=torch.float32, device=self.device))

    def train_step(self, transitions, policy, use_gpi=True, variant=1, beta=1.0, host_losses=None):
        """
        One fused SF TD update.  policy = int -> sequential semantics (sfdqn.py:303-371 / tsfdqn.py:588-709): only that
        policy's (psi, w, g, h) are stepped, next actions by GPI over all policies (use_gpi) or its own psi.
        policy = 'all' -> frozen-snapshot ensemble semantics (agents/sfdqn.py:57-60 batched): every policy is stepped from
        the same pre-step library; with use_gpi every policy i gets a* = argmax_a max_j psi_j(s',a).w_i.
        variant: 0 = G1 (l1 only, 5-tuple), 1 = G2, 2 = G3 (TSF).  Returns losses [n_pol][3] = (loss, l1, l2) on device
        (no host sync; the buffer is one slot of a 64-deep ring, valid for the next 63 steps).
        host_losses: optional CPU float32 tensor with >= n_pol * 3 elements (pinned for a truly asynchronous copy): the step's
        command list then ends with a device-to-host copy of the losses into it -- synchronise the stream before reading.
        """
        if variant == 0:
            states, actions, phis, next_states, gammas = transitions
            rs = None
        else:
            states, actions, rs, phis, next_states, gammas = transitions
        sp = self.spec
        S, D = sp.dims[0], sp.n_features
        states, next_states = self._as_input(states, torch.float32), self._as_input(next_states, torch.float32)
        phis, gammas = self._as_input(phis, torch.float32), self._as_input(gammas, torch.float32)
        actions = self._as_input(actions, torch.int64)
        if states.dim() == 1:
            states, next_states = states.unsqueeze(0), next_states.unsqueeze(0)
        B = states.shape[0]
        if states.dim() != 2 or states.shape[1] != S:
            raise ValueError(f'expected states of shape [B, {S}], got {tuple(states.shape)}')
        if rs is not None:
            rs = self._as_input(rs, torch.float32)
            if rs.numel() != B:
                raise ValueError('rs must hold one reward per transition')
        if not (tuple(next_states.shape) == (B, S) and phis.numel() == B * D and phis.shape[0] == B and gammas.numel() == B
                and actions.numel() == B):
            raise ValueError('inconsistent transition batch shapes')
        if variant == 2 and self.G is None:
            raise Exception('Affine Function (h) is not initialized')          # tsfdqn.py:592-593
        key = ('plan', B, policy, bool(use_gpi), variant, float(beta))
        self.weights_gen += 1
        plan = self._ws.get(key)
        if plan is None:
            plan = self._ws[key] = self._build_plan(B, policy, use_gpi, variant, beta)
            self._build_commands(plan)
        self.last_plan_key = key
        a1, a2, a3, t, b, ad = (plan[k] for k in ('a1', 'a2', 'a3', 't', 'b', 'ad'))
        # inputs: device tensors are read in place; host tensors are staged by H2D commands at the head of the list
        # (host tensors under a one-launch prologue: the prologue kernel pulls pinned ones over PCIe itself -- no copy calls)
        ins = plan['inputs']
        prep = plan.get('prep')
        dptr = []
        for k, src in enumerate((states, actions, rs, phis, next_states, gammas)):
            cmd = plan['h2d'][k]
            cmd.op = 0
            if prep is not None:
                prep.copy_bytes[k] = 0
            if src is None:
                dptr.append(None)
            elif src.is_cuda:
                dptr.append(src.data_ptr())
            elif prep is not None:                            # (pageable sources: sfgpi_step_prep falls back to a plain copy)
                prep.copy_src[k], prep.copy_dst[k] = src.data_ptr(), ins[k].data_ptr()
                prep.copy_bytes[k] = src.numel() * src.element_size()
                dptr.append(ins[k].data_ptr())
            else:
                cmd.op, cmd.p[1] = _lib.OP['H2D'], src.data_ptr()
                dptr.append(ins[k].data_ptr())
        p_states, p_actions, p_rs, p_phis, p_next, p_gammas = dptr
        a1.x, a1.sel_actions = p_states, p_actions
        a2.x = a3.x = p_next
        t.phis, t.gammas, t.states, t.next_states, t.rs = p_phis, p_gammas, p_states, p_next, p_rs
        b.x, b.actions = p_states, p_actions
        if prep is not None:                                  # xo is built in the same launch as the staging copy: read the source
            prep.x = states.data_ptr() if prep.copy_bytes[0] else p_states
        plan['ring'] = (plan['ring'] + 1) % 64
        losses = plan['losses'][plan['ring']]
        ad.losses = losses.data_ptr()
        d2h = plan['d2h_cmd']
        ad.losses_host = None
        if host_losses is None:
            d2h.op = 0
        else:
            if host_losses.is_cuda or host_losses.dtype != torch.float32 or not host_losses.is_contiguous() \
                    or host_losses.numel() < plan['n_pol'] * 3:
                raise ValueError('host_losses must be a contiguous CPU float32 tensor with at least n_pol * 3 elements')
            if host_losses.is_pinned():
                # pinned: the Adam launch's loss block stores the result into the host buffer itself (zero-copy over PCIe) --
                # no copy command between this step's last kernel and the next step's first, their dependent-launch overlap stays
                d2h.op = 0
                ad.losses_host = host_losses.data_ptr()
            else:
                d2h.op, d2h.p[0], d2h.p[1], d2h.i[0] = _lib.OP['D2H'], host_losses.data_ptr(), losses.data_ptr(), plan['n_pol'] * 12
        ad.consts, ad.consts_next = self._adam_consts(plan['lo'], plan['n_pol'])
        peer = plan.get('peer')
        if peer is not None:
            # peer-memory exchange: epoch numbers (identical on every rank) pick the arena halves this step writes / pulls
            pa = self._peer
            pa['ep'][0] += 1
            pa['ep'][1] += 1
            ek, ex = pa['ep']
            koff, xoff = (ek & 1) * peer['kb'], _peer_flag_bytes() + (ex & 1) * pa['xb']
            ka, ua, karena, base = peer['ka'], peer['ua'], peer['karena'], pa['base']
            ka.epoch, ua.epoch = ek, ex
            for r in range(base.world):
                ka.keys_all[r] = karena.ptrs[r] + koff
                ua.x[r] = base.ptrs[r] + xoff
            a2.key_action = karena.local + koff
            if plan['prep'] is not None:
                plan['prep'].keys = karena.local + koff
            else:
                peer['fill_cmd'].p[0] = karena.local + koff
        if plan['tc']:
            for j, which in enumerate(('online', 'online', 'target')):      # the job array embeds copies of the arg blocks
                plan['jobs'][j].args = (a1, a2, a3)[j]
        st = _stream()
        keys, sharded = plan['keys'], plan['sharded']
        segs = plan['segments']
        run = lambda seg: seg[1] and _lib.run(seg[0], seg[1], st, seg[2])
        xc = self._xchg if self._sharded else None
        fused = xc is not None and 'local' in xc              # uniform shards: ONE all-gather per step carries w and h's deltas
        need_h = xc is not None and variant == 2
        if peer is not None:
            if not xc['ok']:                                  # first step (or after outside changes): NCCL gather of w
                self._gather_w(plan['w_all'])
                if peer['nh']:
                    xc['h_prev'].copy_(self.h)
            run(segs[0])                                      # the whole step, exchanges included: one foreign call
            xc['ok'] = True
            return losses
        run(segs[0])                                          # [H2D] pack shadows, key fill
        if sharded and plan['w_all'] is not None and not (fused and xc['ok']):
            self._gather_w(plan['w_all'])                     # first step (or after outside changes): plain gather of w
        run(segs[1])                                          # fold + forwards (fp32: online + GPI forwards)
        if sharded:
            from .dist import allreduce_max_keys
            allreduce_max_keys(keys, self.shard.group)        # packed (value,index) MAX over NVLink: global GPI
        h0 = None
        if need_h:
            if not fused:
                h0 = self.h.clone()
            elif not xc['ok']:
                xc['h_prev'].copy_(self.h)
        run(segs[2])                                          # (fp32: target forward) TD, backward, Adam
        if fused:
            self._exchange(xc, need_h)
        elif h0 is not None:                      # every rank applied only its own optimizers' deltas to the shared h
            import torch.distributed as dist
            delta = self.h - h0
            dist.all_reduce(delta, op=dist.ReduceOp.SUM, group=self.shard.group)
            self.h.copy_(h0 + delta)
        return losses

    def _adam_consts(self, lo, n):
        """
        Adam bias corrections of optimizers [lo, lo+n) for one Adam launch -> (consts, consts_next) pointers.  They are double-
        buffered: the launch reads the current buffer of its optimizers and writes the next step's corrections into the other
        one (no finishing launch).  Optimizers stepped together must be in phase: when they are not (single-policy and
        all-policy steps were mixed), both buffers are refreshed from the step counters first.  Flips their parity.
        """
        par = self._adam_par[lo:lo + n]
        if len(set(par)) > 1:
            _lib.call('sfgpi_adam_refresh', self.step[lo:].data_ptr(), self.adam_consts[lo:].data_ptr(),
                      self.adam_consts2[lo:].data_ptr(), n, 0.9, 0.999, _stream())
            par = [0] * n
        cur, nxt = (self.adam_consts, self.adam_consts2) if par[0] == 0 else (self.adam_consts2, self.adam_consts)
        self._adam_par[lo:lo + n] = [par[0] ^ 1] * n
        return cur[lo:].data_ptr(), nxt[lo:].data_ptr()

    def _exchange(self, xc, with_h):
        """
        End-of-step exchange of a sharded library: x_local = [w_local | h - h_prev] -> all-gather -> w_all (the reward vectors
        the NEXT step's GPI scores against), h = h_prev + sum of every rank's delta, h_prev = h.  Two small kernels around one
        NCCL all-gather replace the w all-gather, the h clone and the delta all-reduce of the unfused path.
        """
        import torch.distributed as dist
        st, D = _stream(), self.spec.n_features
        nw, nh = self.n * D, (xc['nh'] if with_h else 0)
        local, allx = (xc['local'], xc['all']) if nh == xc['nh'] else (xc['local'][:nw], None)
        if allx is None:                                      # TSF library stepped without h (variants 0/1): w only
            allx = xc.setdefault('all_w', self._f(self.shard.world, nw))
        _lib.call('sfgpi_shard_pack', ptr(self.w), nw, ptr(self.h) if nh else None, ptr(xc['h_prev']) if nh else None, nh,
                  ptr(local), st)
        dist.all_gather_into_tensor(allx, local, group=self.shard.group)
        _lib.call('sfgpi_shard_unpack', ptr(allx), self.shard.world, nw, nh, ptr(xc['w_all']), ptr(self.h) if nh else None,
                  ptr(xc['h_prev']) if nh else None, st)
        xc['ok'] = True

    def invalidate_exchange(self):
        """Call after changing w or h of a sharded library from outside train_step (e.g. through the nn.Module views)."""
        if getattr(self, '_xchg', None) is not None:
            self._xchg['ok'] = False

    def _as_input(self, t, dtype):
        """Transition field as a contiguous tensor of `dtype` WITHOUT moving it: host inputs are staged by the command list."""
        if not isinstance(t, torch.Tensor):
            t = torch.as_tensor(t)
        if t.dtype != dtype:
            t = t.to(dtype)
        if t.is_cuda and t.device != self.device:
            t = t.to(self.device)
        return t if t.is_contiguous() else t.contiguous()

    def _build_commands(self, plan):
        """Command lists of one train step (replayed through sfgpi_run): 3 segments, split only where a collective may sit."""
        sp, ws = self.spec, plan['ws']
        B, n_pol = plan['B'], plan['n_pol']
        S, D = sp.dims[0], sp.n_features
        OP = _lib.OP
        dev = self.device
        plan['inputs'] = [torch.empty(B, S, dtype=torch.float32, device=dev), torch.empty(B, dtype=torch.int64, device=dev),
                          torch.empty(B, dtype=torch.float32, device=dev), torch.empty(B, D, dtype=torch.float32, device=dev),
                          torch.empty(B, S, dtype=torch.float32, device=dev), torch.empty(B, dtype=torch.float32, device=dev)]
        plan['desc'] = sp.desc()
        a1, a2, a3, t, b, ad = (plan[k] for k in ('a1', 'a2', 'a3', 't', 'b', 'ad'))
        keys = plan['keys']
        seg0, seg1, seg2 = [], [], []

        def cmd(seg, op, p=(), i=()):
            seg.append((op, list(p), list(i)))

        for k in range(6):
            cmd(seg0, 'NOP', (plan['inputs'][k].data_ptr(), 0), (plan['inputs'][k].numel() * plan['inputs'][k].element_size(),))
        peer = plan.get('peer')
        n_keys = keys.numel() if peer is None else peer['kb'] // 8
        keys_ptr = keys.data_ptr() if peer is None else peer['karena'].local      # peer: patched per step (epoch parity)
        # one-launch prologue (sfgpi_step_prep) whenever nothing has to happen between the packs and the fold, i.e. always
        # except on the NCCL-collective sharded path, whose first steps gather w between them
        st_mode = plan['st']
        merged = plan['tc'] and not st_mode and not (plan['sharded'] and peer is None)
        plan['prep'] = None
        if plan['tc']:
            dref = C.addressof(plan['desc'])
            nw = 1 if a2.w_diag else a2.n_w
            nq = _lib.lib().sfgpi_gpi_fold_rows(C.byref(plan['desc']), nw)
            plan['wq'] = torch.empty(self._parts * a2.n_pol * nq * 256, dtype=torch.float32, device=dev) if st_mode else \
                torch.empty(a2.n_pol * nq * 256, dtype=torch.bfloat16, device=dev)
            plan['bq'] = self._f(a2.n_pol * nq)
        if merged:
            pr = plan['prep'] = _lib.StepPrepArgs()
            pr.net = sp.desc()
            pr.pack_params[0], pr.pack_out[0] = self.online.data_ptr(), self._shadow_for('online').data_ptr()
            pr.pack_lo[0], pr.pack_n[0] = 0, self.n
            pr.pack_params[1], pr.pack_out[1] = self.target.data_ptr(), self._shadow_for('target').data_ptr()
            pr.pack_lo[1], pr.pack_n[1] = a3.policy_lo, a3.n_pol
            pr.keys, pr.n_keys = keys_ptr, n_keys
            pr.fold_params, pr.fold_lo, pr.fold_n = self.online.data_ptr(), a2.policy_lo, a2.n_pol
            pr.w, pr.n_w, pr.w_diag = a2.w, a2.n_w, a2.w_diag
            pr.wq, pr.bq = plan['wq'].data_ptr(), plan['bq'].data_ptr()
            pr.B, pr.xo_bf16 = B, ws['xo'].data_ptr()         # pr.x = this step's states, patched per step
            b.xo_ready = 1
            if t.variant == 2:                                # M = Wh Wg, c once per policy here, not once per CTA of the TD kernel
                if ws.get('tsf_mc') is None:
                    ws['tsf_mc'] = self._f(n_pol, D * S + D)
                pr.tsf_g, pr.tsf_g_stride, pr.tsf_h, pr.tsf_G = self.g.data_ptr(), self.g.shape[1], self.h.data_ptr(), self.G
                pr.tsf_lo, pr.tsf_n, pr.tsf_mc = plan['lo'], n_pol, ws['tsf_mc'].data_ptr()
                t.tsf_mc = ws['tsf_mc'].data_ptr()
            cmd(seg0, 'STEP_PREP', (C.addressof(pr),))
        else:
            if st_mode:
                sh_t, wo_t = self._shadow_t()
                on_sh, tg_sh = self._shadow_for('online').data_ptr(), self._shadow_for('target').data_ptr()
                if a1.n_pol == self.n:      # every policy is stepped: one pack writes the forward AND the transposed (dgrad) operands
                    cmd(seg0, 'PACK_F32', (dref, self.online.data_ptr(), on_sh, sh_t.data_ptr(), wo_t.data_ptr()), (0, self.n, self.cap, self._prec))
                else:                       # GPI reads all policies' forward operands, the dgrad chain only the stepped one's
                    cmd(seg0, 'PACK_F32', (dref, self.online.data_ptr(), on_sh, 0, 0), (0, self.n, self.cap, self._prec))
                    cmd(seg0, 'PACK_F32', (dref, self.online.data_ptr(), on_sh, sh_t.data_ptr(), wo_t.data_ptr()),
                        (a1.policy_lo, a1.n_pol, self.cap, self._prec))
                cmd(seg0, 'PACK_F32', (dref, self.target.data_ptr(), tg_sh, 0, 0), (a3.policy_lo, a3.n_pol, self.cap, self._prec))
            elif plan['tc']:
                cmd(seg0, 'PACK_BF16', (dref, self.online.data_ptr(), self._shadow_for('online').data_ptr()), (0, self.n))
                cmd(seg0, 'PACK_BF16', (dref, self.target.data_ptr(), self._shadow_for('target').data_ptr()), (a3.policy_lo, a3.n_pol))
            cmd(seg0, 'KEYS_FILL', (keys_ptr,), (n_keys,))
            if st_mode:
                cmd(seg1, 'FOLD_GPI_F32', (dref, self.online.data_ptr(), a2.w, plan['wq'].data_ptr(), plan['bq'].data_ptr()),
                    (a2.policy_lo, a2.n_pol, a2.n_w | (a2.w_diag << 31), self._prec))
            elif plan['tc']:
                cmd(seg1, 'FOLD_GPI', (dref, self.online.data_ptr(), a2.w, plan['wq'].data_ptr(), plan['bq'].data_ptr()),
                    (a2.policy_lo, a2.n_pol, a2.n_w, a2.w_diag))
        if plan['tc']:
            jobs = plan['jobs'] = (_lib.ForwardTcJob * 3)()
            for j, which in enumerate(('online', 'online', 'target')):
                jobs[j].params_bf16, jobs[j].n_policies_total = self._shadow_for(which).data_ptr(), self.cap
            jobs[1].wq, jobs[1].bq = plan['wq'].data_ptr(), plan['bq'].data_ptr()
            cmd(seg1, 'NOP')                                  # probe slot (set_probe): event before the dominant kernel
            if st_mode:
                cmd(seg1, 'FORWARD_STREAM', (C.addressof(jobs),), (3, self._prec))
            else:
                cmd(seg1, 'FORWARD_TC_JOBS', (C.addressof(jobs),), (3,))
            cmd(seg1, 'NOP')                                  # probe slot: event after it
        else:
            cmd(seg1, 'FORWARD', (C.addressof(a1),))
            cmd(seg1, 'NOP')
            cmd(seg1, 'FORWARD', (C.addressof(a2),))
            cmd(seg1, 'NOP')
            cmd(seg2, 'FORWARD', (C.addressof(a3),))
        cmd(seg2, 'TD', (C.addressof(t),))
        cmd(seg2, plan['b_op'], (C.addressof(b),))
        cmd(seg2, 'ADAM', (C.addressof(ad),))
        cmd(seg2, 'NOP', (0, 0), (0, 0, 0, 777))              # slot of the optional D2H read-back of the losses (host_losses)
        if peer is not None:
            # peer mode: the exchanges are kernels of the chain -> the sharded step is ONE command list again
            pa, xc = self._peer, self._xchg
            nw, nh = self.n * D, (xc['nh'] if plan['variant'] == 2 else 0)
            ka, ua = _lib.PeerKeysArgs(), _lib.PeerUnpackArgs()
            ka.ctx = ua.ctx = pa['base'].ctx()
            ka.row_lo, ka.n_rows, ka.B, ka.keys_out = peer['lo'], n_pol, B, keys.data_ptr()
            ua.nw, ua.nh, ua.w_all = nw, nh, xc['w_all'].data_ptr()
            if nh:
                ua.h, ua.h_prev = self.h.data_ptr(), xc['h_prev'].data_ptr()
            peer.update(ka=ka, ua=ua, nh=nh)
            n_fill = len(seg0) - 1
            n_keys = len(seg0) + len(seg1)
            if plan['tc']:
                t.peer_keys = C.addressof(ka)                 # the TD kernel pulls the keys of its rows from the peers itself
            else:
                cmd(seg1, 'PEER_KEYS', (C.addressof(ka),))    # fp32 mode: the target forward reads the reduced keys
            ua.pack_w = self.w.data_ptr()                     # x_local is packed by the unpack launch's signalling CTA
            cmd(seg2, 'PEER_UNPACK', (C.addressof(ua),))
            segs = [seg0 + seg1 + seg2, [], []]
        else:
            segs = [seg0, seg1, seg2] if plan['sharded'] else [seg0 + seg1 + seg2, [], []]
        plan['segments'], plan['h2d'], plan['probe'] = [], None, []
        for seg in segs:
            arr = (_lib.Cmd * max(1, len(seg)))()
            launches = 0
            for k, (op, p, i) in enumerate(seg):
                arr[k].op = OP.get(op, 0)
                for q, v in enumerate(p):
                    arr[k].p[q] = v
                for q, v in enumerate(i):
                    arr[k].i[q] = int(v)
                launches += _lib.OP_LAUNCHES[arr[k].op] - (1 if op == 'BACKWARD_TC' and b.xo_ready else 0) - (1 if op == 'ADAM' else 0) \
                    + (1 if op == 'TD' and t.variant == 2 and not t.defer_expand else 0) \
                    + (_lib.lib().sfgpi_step_prep_launches(C.addressof(plan['prep'])) - 1 if op == 'STEP_PREP' else 0)
            if plan['h2d'] is None:
                plan['h2d'] = [arr[k] for k in range(6)]
            plan['probe'] += [arr[k] for k, (op, p, i) in enumerate(seg) if op == 'NOP' and not p]
            for k, (op, p, i) in enumerate(seg):
                if op == 'NOP' and len(i) == 4 and i[3] == 777:
                    plan['d2h_cmd'] = arr[k]
            plan['segments'].append((arr, len(seg), launches))
        if peer is not None:
            arr = plan['segments'][0][0]
            peer['fill_cmd'] = arr[n_fill]

    def set_probe(self, plan_key, start_event=None, end_event=None):
        """
        Measurement hook: record two CUDA events (torch.cuda.Event, timing enabled) around the dominant kernel of a built
        train-step plan -- the fused forward launch -- on every replay, so a benchmark can time that kernel live inside its
        timed region.  Pass None to remove the probes.
        """
        plan = self._ws[plan_key]
        for cmd, ev in zip(plan['probe'][:2], (start_event, end_event)):
            if ev is None:
                cmd.op = 0
            else:
                ev.record()                                   # materialise the lazily created cudaEvent_t
                cmd.op, cmd.p[0] = _lib.OP['EVENT'], ev.cuda_event

    def psi_gradients(self, states, actions, d_out, lo=0, n_pol=None):
        """
        Gradient of sum_{p,b,d} psi_p(s_b)[a_b, d] * d_out[p, b, d] w.r.t. every psi parameter: the backward pass of the train
        step on its own (what autograd computes at sfdqn.py:345 for a given dLoss/dpsi).  Returns [n_pol][row_stride] fp32 in
        library row layout.  Runs the online forward (saving activations) and the backward kernels of the current precision mode.
        """
        x = self._check_x(states)
        n_pol = self.n - lo if n_pol is None else n_pol
        B, D = x.shape[0], self.spec.n_features
        actions = torch.as_tensor(actions).to(device=self.device, dtype=torch.int64).reshape(-1).contiguous()
        d_out = torch.as_tensor(d_out).to(device=self.device, dtype=torch.float32).contiguous()
        if d_out.shape != (n_pol, B, D) or actions.numel() != B:
            raise ValueError('d_out must be [n_pol, B, D] and actions [B]')
        ws = self._workspace(B, n_pol)
        if self.precision != 'fp32':                      # the forward's operands and the backward's (tf32: transposed)
            self._pack('online', lo, n_pol, transposed=True)
        a1 = self._fwd_args(self.online, lo, n_pol, x)
        a1.sel_actions, a1.sel_out = actions.data_ptr(), ptr(ws['cur_sel'])
        self._save_acts(a1, ws['acts'], ws['masks'])
        self._forward(a1, 'online', fresh=True)
        b, entry, _ = self._backward_args(ws, lo, n_pol, B)
        b.x, b.actions, b.d_out = x.data_ptr(), actions.data_ptr(), d_out.data_ptr()
        _lib.call(entry, C.byref(b), _stream())
        return ws['grad_part'].sum(dim=1)

    def train_step_g4(self, transitions, policy, phi_lib, w_bias, coef, use_gpi=True):
        """
        G4 joint psi / phi step (features/deep_phi.py:95-224): phi = phi_theta(cat[s, a, s']) feeds the TD target AND the reward
        fit, loss = phi_loss + coef * psi_loss, one FRESH Adam per call over (psi_i, phi_theta, fit_w[i] incl. bias, coef with
        maximize=True), coef clamped to [1e-2, 1e6].  phi_lib: the one-row PackedSFLibrary holding phi_theta (A = 1, D features);
        w_bias / coef: 1-element fp32 device tensors (updated in place).  Runs on the fp32 CUDA-core kernels (the phi net's
        widths are not the tensor-core shape and the step is launch-latency-bound at the agents' batch 32).
        Returns losses [4] on the device: (loss, psi_loss, phi_loss, coef before the step).
        """
        states, actions, rs, _, next_states, gammas = transitions
        sp = self.spec
        S, D, A = sp.dims[0], sp.n_features, sp.n_actions
        f32 = lambda t: self._as_input(t, torch.float32).to(self.device)
        states, next_states, rs, gammas = f32(states), f32(next_states), f32(rs).reshape(-1), f32(gammas).reshape(-1)
        actions = self._as_input(actions, torch.int64).to(self.device).reshape(-1)
        B = states.shape[0]
        if tuple(states.shape) != (B, S) or tuple(next_states.shape) != (B, S) or rs.numel() != B or gammas.numel() != B or actions.numel() != B:
            raise ValueError('inconsistent transition batch shapes')
        i = int(policy)
        if not (0 <= i < self.n):
            raise IndexError('policy index out of range')
        self.weights_gen += 1
        psp = phi_lib.spec
        if psp.n_features != D or psp.n_actions != 1:
            raise ValueError('the phi network must map cat[s, a, s\'] to n_features values')
        st = _stream()
        ws = self._ws.get(('g4', B))
        if ws is None:
            z = lambda *shape: torch.zeros(*shape, dtype=torch.float32, device=self.device)
            ws = self._ws[('g4', B)] = dict(psi=self._fp32_scratch(1, B), phi=phi_lib._fp32_scratch(1, B), cur=z(1, B, D),
                                            nxt=z(1, B, D), phi_out=z(B, D), d_psi=z(1, B, D), d_phi=z(1, B, D), small=z(D + 2),
                                            losses=z(64, 4), ring=0, keys=torch.empty(1, B, dtype=torch.int64, device=self.device),
                                            zeros=torch.zeros(B, dtype=torch.int64, device=self.device))
        # (1) phi = phi_theta(cat[s, a, s'])                                              deep_phi.py:110-111
        x_phi = torch.cat([states, actions.reshape(B, 1).to(torch.float32), next_states], dim=1).contiguous()
        ap = phi_lib._fwd_args(phi_lib.online, 0, 1, x_phi)
        ap.psi_out = ptr(ws['phi_out'])
        phi_lib._save_acts(ap, ws['phi']['acts'], ws['phi']['masks'])
        _lib.call('sfgpi_mlp_forward', C.byref(ap), st)
        # (2) next actions: GPI over the library under fit_w[i] (the bias shifts every q equally), or the policy's own psi  :113-123
        keys = ws['keys']
        _lib.call('sfgpi_keys_fill', ptr(keys), B, st)
        a2 = self._fwd_args(self.online, 0 if use_gpi else i, self.n if use_gpi else 1, next_states)
        a2.w, a2.n_w, a2.w_diag = C.c_void_p(self.w[i].data_ptr()), 1, 0
        a2.key_action = ptr(keys)
        _lib.call('sfgpi_mlp_forward', C.byref(a2), st)
        # (3) online psi_i(s): saves activations, gathers psi(s)[a];  (4) target psi^-_i(s')[a*]                      :130-136
        a1 = self._fwd_args(self.online, i, 1, states)
        self._save_acts(a1, ws['psi']['acts'], ws['psi']['masks'])
        a1.sel_actions, a1.sel_out = actions.data_ptr(), ptr(ws['cur'])
        _lib.call('sfgpi_mlp_forward', C.byref(a1), st)
        a3 = self._fwd_args(self.target, i, 1, next_states)
        a3.sel_keys, a3.sel_key_stride, a3.sel_out = ptr(keys), B, ptr(ws['nxt'])
        _lib.call('sfgpi_mlp_forward', C.byref(a3), st)
        # (5) losses, d_psi, d_phi, gradients of (w, b, coef)
        ws['ring'] = (ws['ring'] + 1) % 64
        losses = ws['losses'][ws['ring']]
        g = _lib.G4Args()
        g.B, g.A, g.D = B, A, D
        g.cur_sel, g.next_sel, g.phi, g.rs, g.gammas = ptr(ws['cur']), ptr(ws['nxt']), ptr(ws['phi_out']), ptr(rs), ptr(gammas)
        g.w, g.bias, g.coef = C.c_void_p(self.w[i].data_ptr()), ptr(w_bias), ptr(coef)
        g.d_psi, g.d_phi, g.grad_small, g.losses = ptr(ws['d_psi']), ptr(ws['d_phi']), ptr(ws['small']), ptr(losses)
        _lib.call('sfgpi_g4_head', C.byref(g), st)
        # (6) backward through psi_i and through phi_theta
        for lib_, w_, x_, acts_, d_, pol in ((self, ws['psi'], states, actions, ws['d_psi'], i),
                                             (phi_lib, ws['phi'], x_phi, ws['zeros'], ws['d_phi'], 0)):
            b = lib_._fp32_backward(w_, pol, 1, B)
            b.x, b.actions, b.d_out = x_.data_ptr(), acts_.data_ptr(), d_.data_ptr()
            _lib.call('sfgpi_mlp_backward', C.byref(b), st)
        # (7) one fresh Adam over the four groups (lr 1e-3 each, :159-172), coefficient clamped (:212-215)
        ad = _lib.AdamArgs()
        ad.n_pol, ad.fresh, ad.sequential_shared = 1, 1, 1
        ad.beta1, ad.beta2, ad.eps = 0.9, 0.999, 1e-8

        def seg(k, param, length, grad, n_part, part_stride, clamp=None):
            s_ = ad.seg[k]
            s_.param, s_.param_stride, s_.m_stride, s_.v_stride = param, length, length, length
            s_.grad_part, s_.grad_pol_stride, s_.grad_part_stride, s_.n_part = grad, n_part * part_stride, part_stride, n_part
            s_.len, s_.lr, s_.weight_decay = length, 1e-3, 0.0
            if clamp is not None:
                s_.clamp_min, s_.clamp_max = clamp
        seg(0, self.online[i].data_ptr(), sp.row_stride, ws['psi']['grad_part'].data_ptr(), ws['psi']['n_split'], sp.row_stride)
        seg(1, phi_lib.online[0].data_ptr(), psp.row_stride, ws['phi']['grad_part'].data_ptr(), ws['phi']['n_split'], psp.row_stride)
        seg(2, self.w[i].data_ptr(), D, ws['small'].data_ptr(), 1, D + 2)
        seg(3, w_bias.data_ptr(), 1, ws['small'].data_ptr() + 4 * D, 1, D + 2)
        seg(4, coef.data_ptr(), 1, ws['small'].data_ptr() + 4 * (D + 1), 1, D + 2, clamp=(1e-2, 1e6))
        ad.n_seg = 5
        _lib.call('sfgpi_adam_step', C.byref(ad), st)
        return losses

    def _gather_w(self, w_all):
        import torch.distributed as dist
        if self.shard.uniform:
            dist.all_gather_into_tensor(w_all, self.w[:self.n].contiguous(), group=self.shard.group)
        else:
            parts = [w_all[sum(self.shard.counts[:r]):sum(self.shard.counts[:r + 1])] for r in range(self.shard.world)]
            dist.all_gather(parts, self.w[:self.n].contiguous(), group=self.shard.group)

    def target_sync(self, i):
        """update_models_weights(psi_model, target_psi_model) (utils/torch.py:31-33): one contiguous D2D row copy."""
        with torch.no_grad():
            self.target[i].copy_(self.online.detach()[i])
