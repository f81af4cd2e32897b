# -*- coding: UTF-8 -*-
"""
bench.py -- headline benchmark of the SF/GPI hot path (contract: ONE JSON line on stdout, printed by rank 0).

Workload (BASELINE.json configs[1], SURVEY section 8d config 2): TSFDQN on Reacher shapes (S=4, A=9, D=12, MLP 256-256
relu, g: 4->100, h: 100->12, beta=1), synthetic replay batch B=4096, 4 source policies PER GPU, GPI next actions.
One "step" = one replay batch on which EVERY policy of the library is updated (fused all-task TD update, frozen-snapshot
semantics) => transitions x tasks = B * N_total SF TD updates per step.  Multi-GPU: policies sharded 4 per GPU (weak
scaling), the batch replicated, GPI's max over policies exchanged as packed int64 keys.

  value        updates/s with the batches already resident in HBM (CUDA events per step, L2 flushed between steps)
  e2e          same metric through the public API (TSFDQN.update_successor_all) from pinned HOST batches, H2D of the batch and
               D2H of the losses inside the timed region (wall clock, synchronised both sides)
  roofline     the dominant kernel timed live inside the timed steps (events recorded by the step's command list)
  parity_mode  the same step in the mode that meets the reference's precision (1e-5), so the ratio can be read at equal precision
  cpu_baseline / --impl reference : the reference's own classes on the host cores when /root/reference/source is present
               (build container), else the CPU oracle port (GPU box); kind says which.  profiles/r02_port_vs_reference.json
               holds the port-vs-reference calibration measured where both exist.
  gpu_eager_baseline : the port's eager-PyTorch op sequence on cuda:0 -- the honest GPU comparator (SURVEY 8d)
  configs      secondary lines for BASELINE configs 1, 4 (i)/(ii), 5 (config 3 = gpi_eval), each with its CPU figure
  shard_check  (world > 1) sharded == unsharded: GPI keys bit-equal, losses / weights within the mode's tolerance

--dump-outputs DIR writes the last timed step's losses and updated parameters as .npy files (seeded inputs: two builds run with
the same arguments can be compared output for output).
"""
import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    'tsfdqn_reacher_b4096': dict(env='reacher', hidden=[256, 256], acts=['relu', 'relu'], gdim=100, beta=1, B=4096, n_local=4),
    # BASELINE config 4 (ii): TSFDQN dissimilar-task sequence, 256 policies in total split over the GPUs (strong scaling),
    # beta = 30 (reacher_dissimilar.cfg:40), every policy stepped on every batch with GPI over all 256
    'tsfdqn_dissimilar_n256': dict(env='reacher', hidden=[256, 256], acts=['relu', 'relu'], gdim=100, beta=30, B=4096, n_total=256),
}
SEED = 1024
REF_SOURCE = '/root/reference/source'          # present in the build container only; the GPU box times the port
PARITY_MODE = 'tf32x3'                         # the tensor-core mode that meets the reference's 1e-5 on psi / q / losses


def flops_per_net_pass(S, hidden, AD):
    dims = [S, hidden[0]] + list(hidden) + [AD]
    return 2 * sum(dims[i] * dims[i + 1] for i in range(len(dims) - 1))


def load_json(name, default=None):
    try:
        with open(os.path.join(ROOT, name)) as f:
            return json.load(f)
    except Exception:
        return default


def load_peaks():
    p = load_json('MEASURED_PEAKS.json')
    if p:
        return dict(hbm=p['hbm_gbs'], tf_burst=p['bf16_tflops'], tf_sust=p['bf16_tflops_sustained'], src='measured')
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src='fallback')


class ClockSampler:
    """nvidia-smi sampler running DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '20'], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], r[2:6]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons), 'samples': len(sm)}


# ======================================================================================================================
# CPU arm: the reference's own classes (kind "reference") when its sources are present, else the oracle port (kind "port")
# ======================================================================================================================
def env_shapes(cfg):
    from deep_successor_features_for_transfer_b200.workloads import ENVS
    return ENVS[cfg['env']]


class CpuArm:
    """
    The same update, the way the reference does it, on `device` (cpu, or cuda:0 for the eager-GPU comparator):
      kind 'reference' -- tsfdqn.TSFDQN / sfdqn.DeepSF imported UNMODIFIED from /root/reference/source (recipe: SURVEY appendix A);
      kind 'port'      -- oracle/sf_oracle.py (the checker's restatement, the only option where the sources are absent).
    variant 'g3': TSFDQN.update_successor (tsfdqn.py:588-709); 'g2': DeepSF.update_successor (sfdqn.py:303-371).
    """

    def __init__(self, cfg, n_policies, variant='g3', device='cpu', prefer_reference=True):
        shp = env_shapes(cfg)
        self.cfg, self.n, self.variant, self.device = cfg, n_policies, variant, torch.device(device)
        self.S, self.A, self.D = shp['S'], shp['A'], shp['D']
        self.kind = 'port'
        if prefer_reference and self.device.type == 'cpu' and os.path.isdir(REF_SOURCE):
            try:
                self._build_reference()
                self.kind = 'reference'
                return
            except Exception as e:                                   # fall back to the port, say why
                self.why_port = f'{type(e).__name__}: {e}'
        self._build_port()

    def _build_reference(self):
        import types
        from deep_successor_features_for_transfer_b200.workloads import HYPER, ShapeTask
        for m in ('matplotlib', 'matplotlib.pyplot'):
            sys.modules.setdefault(m, types.ModuleType(m))
        sys.modules['matplotlib'].pyplot = sys.modules['matplotlib.pyplot']
        if REF_SOURCE not in sys.path:
            sys.path.insert(0, REF_SOURCE)
        with contextlib.redirect_stdout(io.StringIO()):
            from utils.torch import set_torch_device, get_activation
            from utils.logger import set_logger_level
            set_torch_device(use_gpu=False)
            set_logger_level(use_logger=False)
            import sfdqn as ref_sfdqn
            import tsfdqn as ref_tsfdqn
        cfg = self.cfg
        from collections import OrderedDict

        def sf_model_lambda(num_inputs, output_dim, reshape_dim, reshape_axis=1):      # main_tsfdqn_sequential_torch.py:44-75
            layers = OrderedDict()
            layers['layer_input'] = torch.nn.Linear(num_inputs, cfg['hidden'][0])
            for index, (n, act) in enumerate(zip(cfg['hidden'], cfg['acts'])):
                layers[f'layer_{index}'] = torch.nn.Linear(n, n)
                layers[f'activation_layer_{index}'] = get_activation(act)()
            layers['layer_output'] = torch.nn.Linear(cfg['hidden'][-1], output_dim)
            layers['layer_unflatten'] = torch.nn.Unflatten(reshape_axis, reshape_dim)
            return torch.nn.Sequential(layers), torch.nn.MSELoss(), None

        hyper = dict(HYPER, g_h_function_dims=cfg.get('gdim', 100), beta_loss_coefficient=cfg.get('beta', 1))
        torch.manual_seed(SEED)
        with contextlib.redirect_stdout(io.StringIO()):
            if self.variant == 'g3':
                dsf = ref_tsfdqn.DeepTSF(pytorch_model_handle=sf_model_lambda, use_true_reward=False, target_update_ev=10 ** 9,
                                         hyperparameters=hyper)
                ag = ref_tsfdqn.TSFDQN(deep_sf=dsf, buffer_handle=lambda: ref_tsfdqn.ReplayBuffer(), gamma=0.9, T=500, encoding=None,
                                       use_gpi=True, hyperparameters=hyper)
                ag.reset()
                for i in range(self.n):
                    ag.add_training_task(ShapeTask(self.S, self.A, self.D, i))
                self._step = lambda tr, i, use_gpi: ag.update_successor(tr, i, use_gpi)
                self._gpi = lambda x, i: dsf.GPI(x, i)
            else:
                sf = ref_sfdqn.DeepSF(pytorch_model_handle=sf_model_lambda, use_true_reward=False, target_update_ev=10 ** 9,
                                      hyperparameters=hyper)
                sf.reset()
                for i in range(self.n):
                    sf.add_training_task(ShapeTask(self.S, self.A, self.D, i))
                self._step = lambda tr, i, use_gpi: sf.update_successor(tr, i, use_gpi)
                self._gpi = lambda x, i: sf.GPI(x, i)

    def _build_port(self):
        from oracle.sf_oracle import OracleSF
        cfg = self.cfg
        gen = torch.Generator().manual_seed(SEED)
        o = OracleSF(self.S, self.A, self.D, cfg['hidden'], cfg['acts'], tsf_dim=cfg.get('gdim', 100) if self.variant == 'g3' else None,
                     beta=cfg.get('beta', 1), target_update_ev=10 ** 9)
        for _ in range(self.n):
            o.add_random_policy(gen)
        if self.device.type != 'cpu':
            o.to(self.device)
        self._step = (lambda tr, i, use_gpi: o.tsf_update_successor(tr, i, use_gpi)) if self.variant == 'g3' else \
            (lambda tr, i, use_gpi: o.update_successor(tr, i, use_gpi))
        self._gpi = lambda x, i: o.GPI(x, i)

    def batches(self, B, n=2, hopper=False):
        from deep_successor_features_for_transfer_b200.workloads import synthetic_transitions
        gen = torch.Generator().manual_seed(SEED + 1)
        return [tuple(t.to(self.device) for t in synthetic_transitions(B, self.S, self.A, self.D, gen, hopper=hopper)) for _ in range(n)]

    def sync(self):
        if self.device.type == 'cuda':
            torch.cuda.synchronize(self.device)

    def time_steps(self, B, policies, steps, warmup, use_gpi=True):
        """`steps` x (one update_successor call per policy in `policies` on the same batch); returns seconds per step."""
        batches = self.batches(B)
        with contextlib.redirect_stdout(io.StringIO()):
            for k in range(warmup):
                for i in policies:
                    self._step(batches[k % 2], i, use_gpi)
            self.sync()
            t0 = time.perf_counter()
            for k in range(steps):
                for i in policies:
                    self._step(batches[k % 2], i, use_gpi)
            self.sync()
        return (time.perf_counter() - t0) / steps

    def time_gpi(self, B, reps, hopper=False):
        x = self.batches(B, 1, hopper=hopper)[0][4]
        with torch.no_grad():
            self._gpi(x, 0)
            self.sync()
            t0 = time.perf_counter()
            for _ in range(reps):
                self._gpi(x, 0)
            self.sync()
        return (time.perf_counter() - t0) / reps


def cpu_all_task(cfg, n_total, steps, warmup, threads, prefer_reference=True):
    """The all-task update the way the reference does it: one update_successor per task on the same batch."""
    torch.set_num_threads(threads)
    arm = CpuArm(cfg, n_total, 'g3', 'cpu', prefer_reference)
    per = arm.time_steps(cfg['B'], list(range(n_total)), steps, warmup)
    return cfg['B'] * n_total / per, per, arm.kind


def run_reference(args, cfg, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n_total = cfg['n_local'] * world
    # every step = n_total update_successor calls, each with GPI over n_total nets: bound the run to a few minutes
    est = 0.012 * n_total * (n_total + 4)                           # ~12 ms per net pass-batch on 16 cores (B = 4096)
    steps = max(1, min(args.steps, int(120 / max(est, 1e-3)) or 1))
    warm = max(1, min(args.warmup, 2))
    val, per, kind = cpu_all_task(cfg, n_total, steps, warm, cores)
    sample = (f'{steps} all-task steps ({n_total} update_successor calls each) of the same workload, B={cfg["B"]}'
              + ('' if steps == args.steps else f' (--steps {args.steps} capped so that the run ends within minutes)'))
    cal = load_json('profiles/r02_port_vs_reference.json')
    print(json.dumps({
        'impl': 'reference', 'metric': 'SF TD updates (transitions x tasks)/s', 'value': val, 'unit': 'updates/s',
        'n_gpus': world, 'steps': steps, 'warmup': warm, 'ms_per_step': per * 1e3, 'higher_is_better': True,
        'scaling': 'strong' if 'n_total' in cfg else 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args.workload, cfg, n_total, world, args.l2),
        'cpu_baseline': {'value': val, 'unit': 'updates/s', 'cores': cores, 'kind': kind, 'sample': sample,
                         'port_vs_reference': cal if kind == 'port' else None},
        'e2e': {'value': val, 'unit': 'updates/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


def workload_config(name, cfg, n_total, world, l2='flush', exchange=None):
    """The workload only (identical for both arms): precision / transport are reported outside `config`."""
    shp = env_shapes(cfg)
    return {'workload': f'{name}: TSFDQN {cfg["env"]} S{shp["S"]}/A{shp["A"]}/D{shp["D"]} MLP 256-256 relu, g {shp["S"]}->100, h 100->{shp["D"]}, '
                        f'beta={cfg["beta"]}, B={cfg["B"]}, {cfg["n_local"]} policies/GPU ({n_total} total), all-task TD update with GPI next actions',
            'batch': cfg['B'], 'policies_total': n_total, 'policies_per_gpu': cfg['n_local'],
            'parallelism': f'policy-sharded x{world}' if world > 1 else 'single GPU',
            'l2': ('flushed between timed steps (256 MiB write), flush excluded from the per-step CUDA-event time' if l2 == 'flush'
                   else 'inputs larger than L2: >160 MB of distinct resident batches cycled, weights / optimizer state stay '
                        'L2-resident as in a real training loop (--l2 flush: 256 MiB write between per-step brackets)')}


PRECISION_TEXT = {
    'bf16': 'bf16 operands on tcgen05 in every psi GEMM (forwards AND dgrad / wgrad), fp32 accumulate in TMEM, fp32 master weights, '
            'fp32 TD / g / h gradients / Adam (stated tolerance: 2e-2 on psi / q, K-step bounds in tests/test_gpu_bf16.py)',
    'fp32': 'fp32 CUDA-core FFMA kernels (1e-5 parity mode)',
    'tf32': 'tf32 operands on tcgen05 (kind::tf32), fp32 accumulate (stated tolerance 2e-3)',
    'tf32x3': '3-pass split tf32 on tcgen05 (a_hi.b_hi + a_hi.b_lo + a_lo.b_hi, fp32 accumulate in TMEM): 1e-5 parity mode on the tensor cores',
}


# ======================================================================================================================
# GPU arm
# ======================================================================================================================
class Timer:
    """CUDA-event timing of a callable, L2 flushed between iterations (flush outside the events)."""

    def __init__(self, dev):
        self.dev = dev
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def run(self, fn, steps, warmup, flush=True):
        for k in range(warmup):
            fn(k)
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for k in range(steps):
            if flush:
                self.flush.fill_(k & 0xFF)
            ev[k][0].record()
            fn(warmup + k)
            ev[k][1].record()
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in ev]


def build_agent(cfg, n_local, precision, first_policy=0):
    from deep_successor_features_for_transfer_b200.workloads import build_tsf_agent
    return build_tsf_agent(cfg['env'], n_local, cfg['hidden'], cfg['acts'], cfg['gdim'], cfg['beta'], precision, True,
                           seed=SEED + 10, first_policy=first_policy)


GPI_EVAL = dict(env='hopper', hidden=[256, 256], acts=['relu', 'relu'], N=64, B=65536)


def time_gpi_eval(world, rank, dev, precision, barrier, reps=10):
    from deep_successor_features_for_transfer_b200.workloads import build_sf_library, ENVS
    import torch.distributed as dist
    c = GPI_EVAL
    shp = ENVS[c['env']]
    if c['N'] % world:
        return {'skipped': f'{c["N"]} policies do not split over {world} ranks'}
    n_local = c['N'] // world
    sf = build_sf_library(c['env'], n_local, c['hidden'], c['acts'], precision, seed=SEED + 100, first_policy=rank * n_local)
    lib = sf._library
    if world > 1:
        lib.enable_sharding()
    gen = torch.Generator().manual_seed(SEED + 7)
    x = torch.sigmoid(torch.randn(c['B'], shp['S'], generator=gen)).to(dev)          # tasks/hopper_phi.py:59
    w = torch.empty(shp['D']).uniform_(-0.01, 0.01, generator=gen).to(dev)           # sfdqn.py:197
    for _ in range(3):
        lib.gpi(x, w, want_q=False)
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        _, ka, kt = lib.gpi(x, w, want_q=False)
        b.record()
    barrier()
    ms = torch.tensor([sum(a.elapsed_time(b) for a, b in ev) / reps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms)
    best_action, best_val = lib.decode_keys(ka, want_value=True)                      # the result a caller reads
    # self-check against an independent path of the same library: q of 256 spot states from the psi form (get_successors . w)
    spot = torch.arange(0, c['B'], c['B'] // 256, device=dev)[:256]
    psi = lib.forward_psi(x[spot])                                                    # [256][n_local][A][D]
    q = (psi * w.view(1, 1, 1, -1)).sum(-1)                                           # local policies only
    qmax = q.reshape(256, -1).max(dim=1).values
    if world > 1:
        dist.all_reduce(qmax, op=dist.ReduceOp.MAX)
    tol = 2e-2 if precision == 'bf16' else 1e-4
    dev_rel = float(((best_val[spot] - qmax).abs() / qmax.abs().max()).max())
    F = flops_per_net_pass(shp['S'], c['hidden'], shp['A'] * shp['D']) + 2 * shp['A'] * shp['D']      # the reference's arithmetic (SURVEY 8d)
    F_exec = flops_per_net_pass(16, c['hidden'], (shp['A'] + 15) // 16 * 16)                         # w folded into the output layer, K0 padded
    return {'metric': 'GPI action evals/s', 'value': c['B'] / (ms * 1e-3), 'unit': 'states/s (each over all 64 policies)',
            'ms_per_eval': ms, 'algorithmic_tflops_per_gpu': n_local * c['B'] * F / (ms * 1e-3) / 1e12,
            'executed_tflops_per_gpu': n_local * c['B'] * F_exec / (ms * 1e-3) / 1e12, 'scaling': 'strong',
            'note': 'algorithmic = N*F per state as the reference computes it (psi[B,N,A,D] then .w); executed = what the kernel '
                    'runs after folding w into the output layer (A columns instead of A*D), so algorithmic can exceed the bf16 peak',
            'config': f'SFDQN Hopper S11/A27/D50, {c["N"]} policies ({n_local}/GPU), B={c["B"]} resident states, pack + fold + fused '
                      f'forward/GPI kernel + key all-reduce per eval',
            'precision': precision,
            'check': {'ok': bool(int(best_action.min()) >= 0 and int(best_action.max()) < shp['A'] and dev_rel < tol),
                      'what': 'max GPI value of 256 spot states vs the psi-form forward (get_successors . w) of the same library',
                      'max_rel_dev': dev_rel, 'tol': tol}}


def measure_steps(cfg, n_local, precision, dev, steps, warmup, timer, single_policy=None, B=None, use_gpi=True, variant='g3',
                  env=None, count_launches=True, with_trace=False):
    """
    Median / mean ms of one train step on a FRESH agent of `precision` (HBM-resident batches, CUDA events, L2 flushed):
    all-task step (single_policy None) or the sequential step of one policy.  variant g2 = DeepSF.update_successor.
    """
    from deep_successor_features_for_transfer_b200 import _lib
    from deep_successor_features_for_transfer_b200.workloads import build_tsf_agent, build_sf_library, synthetic_transitions, ENVS
    c = dict(cfg, env=env or cfg['env'])
    shp = ENVS[c['env']]
    B = B or c['B']
    if variant == 'g3':
        dsf, ag = build_tsf_agent(c['env'], n_local, c['hidden'], c['acts'], c.get('gdim', 100), c.get('beta', 1), precision, True, seed=SEED + 10)
    else:
        dsf = ag = build_sf_library(c['env'], n_local, c['hidden'], c['acts'], precision, seed=SEED + 10)
    gen = torch.Generator().manual_seed(SEED)
    res = [tuple(t.to(dev) for t in synthetic_transitions(B, shp['S'], shp['A'], shp['D'], gen)) for _ in range(8)]
    if single_policy is None:
        fn = lambda k: ag.update_successor_all(res[k % 8], use_gpi=use_gpi)
        n_upd = n_local
    else:
        fn = lambda k: ag.update_successor(res[k % 8], single_policy, use_gpi)
        n_upd = 1
    fn(0)
    l0 = _lib.launch_count
    fn(1)
    launches = _lib.launch_count - l0
    ms = timer.run(fn, steps, warmup)
    med = statistics.median(ms)
    out = {'precision': precision, 'ms_per_step': med, 'ms_per_step_mean': sum(ms) / len(ms), 'steps_timed': steps,
           'value': B * n_upd / (med * 1e-3), 'unit': 'updates/s' if single_policy is None else 'transitions/s'}
    if count_launches:
        out['launches_per_step'] = launches
    if with_trace:                                    # per-kernel windows + the HBM-bound kernels' bandwidth at THIS size
        try:
            out['step_trace'] = trace_steps(fn, n=5)
            out['hbm_kernels'] = hbm_kernels(out['step_trace'], dsf._library, B, n_upd, n_local, load_peaks())
        except Exception as e:
            out['step_trace'] = {'error': f'{type(e).__name__}: {e}'}
    del dsf, ag
    return out


def secondary_configs(args, dev, timer, cores, with_cpu):
    """BASELINE configs 1, 4 (i)/(ii), 5 next to the headline (config 2) and gpi_eval (config 3); one GPU."""
    out = {}
    reacher = dict(env='reacher', hidden=[256, 256], acts=['relu', 'relu'], gdim=100, beta=1, B=4096)
    modes = [args.precision] if args.precision == PARITY_MODE else [args.precision, PARITY_MODE]

    def cpu(cfg, n, variant, B, policies, steps, use_gpi=True):
        if not with_cpu:
            return None
        torch.set_num_threads(cores)
        arm = CpuArm(cfg, n, variant, 'cpu')
        per = arm.time_steps(B, policies, steps, 1, use_gpi)
        return {'ms_per_step': per * 1e3, 'value': B * len(policies) / per, 'cores': cores, 'kind': arm.kind, 'steps_timed': steps}

    # config 1: G2 SFDQN Reacher, N = 4, sequential step of one policy with GPI over the library, B = 32 (reacher.cfg) and 4096
    c1 = {}
    for B in (32, 4096):
        c1[f'B{B}'] = {'gpu': [measure_steps(reacher, 4, m, dev, 200, 20, timer, single_policy=1, B=B, variant='g2') for m in modes],
                       'cpu': cpu(reacher, 4, 'g2', B, [1], 20 if B == 32 else 5)}
    out['config1_sfdqn_reacher_n4'] = dict(c1, what='DeepSF.update_successor(transitions, 1, use_gpi=True) (sfdqn.py:303-371), transitions/s')
    # config 5: G2 at CartPole shapes, N = 3, B = 32, use_gpi = False: latency
    cart = dict(env='cartpole', hidden=[256, 256], acts=['relu', 'relu'], B=32)
    g = [measure_steps(cart, 3, m, dev, 200, 20, timer, single_policy=0, B=32, use_gpi=False, variant='g2') for m in modes]
    for r in g:
        r['us_per_step'] = r['ms_per_step'] * 1e3
    out['config5_cartpole_b32'] = {'gpu': g, 'cpu': cpu(cart, 3, 'g2', 32, [0], 50, use_gpi=False),
                                   'what': 'DeepSF.update_successor(transitions, 0, use_gpi=False) at CartPole shapes S4/A2/D20, N=3, B=32 '
                                           '(cartpole_phi.cfg): latency-bound, us/step and kernel launches per step; phi is synthetic'}
    # config 4: TSFDQN dissimilar, N = 256, beta = 30, B = 4096: (i) one policy stepped with GPI over 256, (ii) all 256 stepped
    if not args.no_config4:
        c4 = dict(reacher, beta=30)
        seq = measure_steps(c4, 256, args.precision, dev, 30, 5, timer, single_policy=7)
        ens = measure_steps(c4, 256, args.precision, dev, 20, 3, timer, with_trace=True)
        c4cpu = cpu(c4, 256, 'g3', 4096, [7], 2)
        if c4cpu is not None:
            c4cpu['ensemble_extrapolated'] = {'ms_per_step': c4cpu['ms_per_step'] * 256, 'value': 4096 * 256 / (c4cpu['ms_per_step'] * 256e-3),
                                              'how': '256 x the sequential step: the reference steps all tasks by looping update_successor '
                                                     'over them (agents/sfdqn.py:59-60), each call re-running GPI over all 256 nets'}
        out['config4_tsfdqn_dissimilar_n256'] = {'sequential_one_policy': seq, 'ensemble_all_policies': ens, 'cpu_sequential': c4cpu,
                                                 'what': 'TSFDQN beta=30, 256 policies, B=4096 on ONE GPU: (i) update_successor(transitions, 7, True) '
                                                         'transitions/s, (ii) update_successor_all updates/s; multi-GPU strong scaling: '
                                                         '--workload tsfdqn_dissimilar_n256 --gpus N'}
    return out


def gpu_eager_baseline(cfg, n_total, dev, steps=3):
    """The reference's eager op sequence (the oracle port, plain tensors) on cuda:0: the fair GPU comparator of SURVEY 8d."""
    arm = CpuArm(cfg, n_total, 'g3', dev, prefer_reference=False)
    per = arm.time_steps(cfg['B'], list(range(n_total)), steps, 2)
    return {'value': cfg['B'] * n_total / per, 'unit': 'updates/s', 'ms_per_step': per * 1e3, 'kind': 'port on cuda:0 (eager PyTorch fp32, TF32 off)',
            'sample': f'{steps} all-task steps ({n_total} update_successor calls each), wall clock with synchronize'}


TRACE_SLOTS = ('prep', 'forward', 'td', 'dgrad', 'wgrad', 'adam')


def trace_steps(step_fn, n=9):
    """
    Kernel windows of n ISOLATED steps from the in-kernel %globaltimer trace (csrc/common.cuh, sfgpi_trace_*): per kernel the
    median of [first CTA past its dependency wait -> last CTA exit] and of the hand-over gap to it (predecessor's last exit ->
    this kernel past its wait), in microseconds.  Unlike a CUDA-event bracket the trace does not sit between two kernels of the
    chain, so their programmatic-dependent-launch overlap stays as it is in the timed steps.
    """
    import ctypes as C
    from deep_successor_features_for_transfer_b200 import _lib
    L = _lib.lib()
    L.sfgpi_trace_enable(1)
    buf = (C.c_uint64 * (3 * 8))()
    rows = []
    try:
        for k in range(n + 2):
            step_fn(k)
            if L.sfgpi_trace_read(buf, 8) == 0:
                return None
            if k >= 2:
                rows.append([int(v) for v in buf])
    finally:
        L.sfgpi_trace_enable(0)
    out, none = {}, (1 << 64) - 1
    for i, name in enumerate(TRACE_SLOTS):
        busy = [(r[3 * i + 2] - r[3 * i + 1]) / 1e3 for r in rows if r[3 * i] != none]
        if not busy:
            continue
        out[name] = {'busy_us': statistics.median(busy)}
        if i > 0:
            gaps = [(r[3 * i + 1] - r[3 * (i - 1) + 2]) / 1e3 for r in rows if r[3 * i] != none and r[3 * (i - 1)] != none]
            if gaps:
                out[name]['handover_us'] = statistics.median(gaps)
    spans = [(max(r[3 * i + 2] for i in range(6)) - min(r[3 * i] for i in range(6) if r[3 * i] != none)) / 1e3 for r in rows]
    out['step_span_us'] = statistics.median(spans)
    out['what'] = ('isolated steps (device synchronised between them: clocks ramp down a little, so these are upper bounds of the '
                   'in-stream times); busy = first CTA past its dependency wait -> last CTA exit; handover = predecessor\'s last '
                   'exit -> this kernel past its wait')
    return out


def hbm_kernels(trace, lib, B, n_pol, n_w, peaks):
    """
    The step's HBM-bound kernels against the measured copy bandwidth: ALGORITHMIC bytes per launch (DESIGN section 3) over the
    in-kernel busy window of the trace.  prologue: fp32 library rows read + bf16 shadow written (online and target: 6 B per
    parameter each), 8 B per GPI key filled, the GPI fold (read the output layer once, write n_w * A folded rows of 256 bf16 per
    policy); TD: 4 B (3 D + 3 + 2 S) per (transition, policy) + the 8-byte key; Adam: 28 B per parameter + 4 B per split-K partial.
    """
    if not trace:
        return None
    sp = lib.spec
    S, A, D = sp.dims[0], sp.n_actions, sp.n_features
    n_split = max([ws.get('n_split', 1) for ws in lib._ws.values() if isinstance(ws, dict)] + [1])
    wb = 8 if n_w >= 8 else (4 if n_w >= 4 else 1)
    fold_rows = (n_w + wb - 1) // wb * wb * A
    by = {'prep': n_pol * (2 * 6 * sp.n_params + 4 * A * D * 256 + 2 * 256 * fold_rows) + 8 * n_w * B,
          'td': n_pol * B * (4 * (3 * D + 3 + 2 * S) + 8),
          'adam': n_pol * sp.n_params * (28 + 4 * n_split)}
    out = {'peak_GBps': peaks['hbm'], 'n_split': n_split,
           'what': 'algorithmic bytes per launch / in-kernel busy window (step_trace), as a fraction of the measured HBM copy bandwidth; '
                   'at the headline size these launches are latency-bound (a few MB in one wave), at config 4 sizes bandwidth matters'}
    for k, b in by.items():
        if k in trace and trace[k].get('busy_us'):
            gbps = b / (trace[k]['busy_us'] * 1e-6) / 1e9
            out[k] = {'bytes': b, 'busy_us': trace[k]['busy_us'], 'GBps': gbps, 'frac': gbps / peaks['hbm']}
    return out


def config4_strong(world, rank, dev, precision, barrier, steps=20, warm=5):
    """
    BASELINE config 4 (ii) on ALL ranks of this run (strong scaling): 256 TSFDQN policies (beta = 30) split over the GPUs, every
    policy stepped on every batch with GPI over all 256 reward vectors.  Secondary line of the multi-GPU runs: the driver's
    scaling sweep launches the default (weak-scaling) workload; this adds the multi-GPU train configuration BASELINE names.
    """
    import torch.distributed as dist
    from deep_successor_features_for_transfer_b200.workloads import synthetic_transitions
    cfg = dict(WORKLOADS['tsfdqn_dissimilar_n256'])
    if cfg['n_total'] % world:
        return {'skipped': f'{cfg["n_total"]} policies do not split over {world} ranks'}
    n_local = cfg['n_total'] // world
    shp = env_shapes(cfg)
    dsf, ag = build_agent(cfg, n_local, precision, first_policy=rank * n_local)
    lib = dsf._library
    if world > 1:
        lib.enable_sharding()
    gen = torch.Generator().manual_seed(SEED)
    res = [tuple(t.to(dev) for t in synthetic_transitions(cfg['B'], shp['S'], shp['A'], shp['D'], gen)) for _ in range(4)]
    for k in range(warm):
        ag.update_successor_all(res[k % 4], use_gpi=True)
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for k in range(steps):
        ev[k][0].record()
        ag.update_successor_all(res[k % 4], use_gpi=True)
        ev[k][1].record()
    barrier()
    ms = torch.tensor([sum(a.elapsed_time(b) for a, b in ev) / steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        lib._close_peer()
    ms = float(ms)
    del dsf, ag
    return {'workload': 'tsfdqn_dissimilar_n256 (BASELINE config 4 ii)', 'ms_per_step': ms, 'value': cfg['B'] * cfg['n_total'] / (ms * 1e-3),
            'unit': 'updates/s', 'scaling': 'strong', 'policies_per_gpu': n_local, 'steps_timed': steps, 'precision': precision,
            'l2': 'not flushed between steps (one step streams > 1 GB)'}


def shard_check(cfg, n_local, precision, rank, world, dev, K=3):
    """
    Driver-side evidence that the policy-sharded step (the path every N > 1 number comes from) computes what one GPU computes:
    fresh sharded agents on every rank and a fresh unsharded agent with all n_total policies on rank 0, built from the same
    per-policy seeds, run the same K all-task steps.  GPI keys of a probe batch before training must be BIT-equal; losses and
    post-step weights agree within the mode's tolerance (the shared h receives the ranks' deltas in a different summation order).
    """
    import torch.distributed as dist
    from deep_successor_features_for_transfer_b200.workloads import synthetic_transitions
    shp = env_shapes(cfg)
    n_total = n_local * world
    gen = torch.Generator().manual_seed(SEED + 5)
    B = 1024
    batches = [tuple(t.to(dev) for t in synthetic_transitions(B, shp['S'], shp['A'], shp['D'], gen)) for _ in range(K)]
    dsf, ag = build_agent(cfg, n_local, precision, first_policy=rank * n_local)
    lib = dsf._library
    lib.enable_sharding()
    w0 = torch.full((shp['D'],), 0.005, device=dev)
    _, ka, kt = lib.gpi(batches[0][4], w0, want_q=False)
    keys = torch.stack([ka, kt]).clone()
    losses = torch.stack([ag.update_successor_all(b, use_gpi=True).clone() for b in batches])          # [K][n_local][3]
    rows = lib.online[:n_local].clone()
    all_losses = [torch.empty_like(losses) for _ in range(world)]
    all_rows = [torch.empty_like(rows) for _ in range(world)]
    dist.all_gather(all_losses, losses)
    dist.all_gather(all_rows, rows)
    h_sh = lib.h.clone()
    res = None
    if rank == 0:
        fdsf, fag = build_agent(cfg, n_total, precision)
        flib = fdsf._library
        _, fka, fkt = flib.gpi(batches[0][4], w0, want_q=False)
        keys_equal = bool(torch.equal(keys[0], fka) and torch.equal(keys[1], fkt))
        fl = torch.stack([fag.update_successor_all(b, use_gpi=True).clone() for b in batches])          # [K][n_total][3]
        sl = torch.cat(all_losses, dim=1)
        dl = float(((fl - sl).abs() / fl.abs().clamp_min(1e-12)).max())
        sr = torch.cat(all_rows, dim=0)
        dw = float((flib.online[:n_total] - sr).abs().max() / flib.online[:n_total].abs().max())
        dh = float((flib.h - h_sh).abs().max() / flib.h.abs().max())
        tol = 5e-5 if precision in ('fp32', 'tf32x3') else 5e-3
        res = {'ok': bool(keys_equal and dl < tol and dw < tol and dh < tol), 'gpi_keys_bit_equal': keys_equal, 'max_rel_dev_losses': dl,
               'max_rel_dev_psi_weights': dw, 'max_rel_dev_h': dh, 'tol': tol, 'steps': K, 'batch': B, 'policies_total': n_total,
               'transport': 'peer-memory kernels' if lib._peer is not None else 'NCCL collectives', 'precision': precision,
               'what': 'sharded (this run\'s path) vs all policies on rank 0: keys of a probe batch before training, then K all-task steps'}
    torch.cuda.synchronize()
    dist.barrier()
    lib._close_peer()
    return res


DUMP_MAX_BYTES = 60 << 20          # --dump-outputs: array data; with the .npy headers the files stay under 64 MB


def step_outputs(losses, lib, n_local):
    """
    What one all-task step computed, as float32 host arrays: the losses update_successor_all returned ([n_local][3]: loss,
    psi loss, phi loss) and the parameters it updated -- the packed online psi rows, w, g of the local policies and the shared h.
    """
    out = {'losses': losses, 'psi_online': lib.online[:n_local], 'w': lib.w[:n_local], 'g': lib.g[:n_local], 'h': lib.h}
    return {k: v.detach().float().cpu().numpy() for k, v in out.items()}


def write_outputs(arrays, dirname, max_bytes=DUMP_MAX_BYTES):
    """
    DIR/<name>.npy per array.  When the arrays hold more than max_bytes in all, the largest ones are cut down to a fixed, seeded
    sample of their elements (flattened, in index order) so the total fits: the same shapes always give the same sample.
    """
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    sizes = {k: a.nbytes for k, a in arrays.items()}
    budget = max_bytes
    for i, k in enumerate(sorted(arrays, key=lambda k: sizes[k])):          # smallest first: each takes at most a fair share
        a = arrays[k]
        share = budget // (len(arrays) - i)
        if a.nbytes > share:
            keep = share // a.itemsize
            idx = np.sort(np.random.default_rng(SEED).choice(a.size, keep, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(dirname, k + '.npy'), a)
        budget -= a.nbytes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='tsfdqn_reacher_b4096')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-gpi-eval', action='store_true', help='skip the secondary M2 measurement (quick A/B runs)')
    ap.add_argument('--no-secondary', action='store_true', help='skip configs 1 / 4 / 5, parity mode, eager-GPU comparator')
    ap.add_argument('--no-config4', action='store_true', help='skip the 256-policy secondary line (builds 256 policies)')
    ap.add_argument('--l2', default='inputs', choices=['flush', 'inputs'],
                    help='flush: 256 MiB write between timed steps (everything cold, weights included); inputs: cycle through '
                         'more distinct resident batches than fit in L2 (inputs cold, weights stay L2-resident)')
    ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp32', 'tf32', 'tf32x3'])
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed (losses, updated parameters; rank 0\'s policies) '
                         'as DIR/<name>.npy, float32, at most 64 MB in all; inputs are seeded, so two builds compare output for output')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    cfg = dict(WORKLOADS[args.workload])
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    strong = 'n_total' in cfg
    if strong:
        if cfg['n_total'] % world:
            raise SystemExit(f'{cfg["n_total"]} policies do not split over {world} ranks')
        cfg['n_local'] = cfg['n_total'] // world
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        run_reference(args, cfg, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3
    import torch.distributed as dist
    from deep_successor_features_for_transfer_b200 import _lib
    from deep_successor_features_for_transfer_b200.workloads import synthetic_transitions
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    shp = env_shapes(cfg)
    B, S, A, D, n_local = cfg['B'], shp['S'], shp['A'], shp['D'], cfg['n_local']
    n_total = n_local * world
    dsf, ag = build_agent(cfg, n_local, args.precision, first_policy=rank * n_local)
    lib = dsf._library
    if world > 1:
        lib.enable_sharding()
    gen = torch.Generator().manual_seed(SEED)                       # identical batches on every rank (replicated replay)
    host = [synthetic_transitions(B, S, A, D, gen) for _ in range(8)]
    pinned = [tuple(t.pin_memory() for t in tr) for tr in host]
    batch_bytes = sum(t.numel() * t.element_size() for t in host[0])
    n_res = 8 if args.l2 == 'flush' else int(160e6 // batch_bytes) + 1        # 'inputs': > 126 MB L2 worth of batches
    resident = [tuple(t.to(dev) for t in host[k % 8]) for k in range(n_res)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- value: HBM-resident inputs, CUDA events per step ----------------
    # nvidia-smi needs ~0.1 s to start and the timed regions last milliseconds: it samples every 20 ms from here (before the
    # warm-up) to the end of the e2e loop, i.e. throughout both timed regions and the loaded phases around them.
    sampler = ClockSampler(local_rank)
    sampler.start()
    n_warm = max(args.warmup, 1000 if not strong else 20)   # a FIXED count (identical on every rank): >= W steps, clocks settled under load
    for k in range(n_warm):
        ag.update_successor_all(resident[k % n_res], use_gpi=True)
    barrier()
    plan_key = lib.last_plan_key
    launches = None
    stream_ms = None
    outputs = None                                                  # --dump-outputs: the last timed step's results
    if args.l2 == 'inputs':
        # The K timed steps as ONE stream of work between two events (inputs larger than L2: n_res distinct resident batches are
        # cycled, > 160 MB): what a training loop sees -- the kernels of consecutive steps chain through programmatic dependent
        # launch, no event sits between them.
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count
        barrier()
        e0.record()
        for k in range(args.steps):
            losses = ag.update_successor_all(resident[(n_warm + k) % n_res], use_gpi=True)
        e1.record()
        barrier()
        launches = _lib.launch_count - l0
        stream_ms = e0.elapsed_time(e1)
        if args.dump_outputs:                                       # before the bracketed steps below move the weights on
            outputs = step_outputs(losses, lib, n_local)
    # per-step brackets: an event pair around every step and probes around the dominant kernel (the one-launch fused forward:
    # online psi(s) + GPI(s') + target psi(s')), recorded by the command list itself inside the step.  'flush' mode: these ARE
    # the timed steps (256 MiB write between them, outside the brackets).
    n_probe = args.steps if args.l2 == 'flush' else min(args.steps, 100)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_probe)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_probe)]
    l0 = _lib.launch_count
    barrier()
    for k in range(n_probe):
        if args.l2 == 'flush':
            flush.fill_(k & 0xFF)
        lib.set_probe(plan_key, *kev[k])
        ev[k][0].record()
        losses = ag.update_successor_all(resident[(n_warm + k) % n_res], use_gpi=True)
        ev[k][1].record()
    barrier()
    lib.set_probe(plan_key, None, None)
    if args.dump_outputs and outputs is None:                       # --l2 flush: these were the timed steps
        outputs = step_outputs(losses, lib, n_local)
    if launches is None:
        launches = _lib.launch_count - l0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    bracket_ms = sum(step_ms) / n_probe
    total_ms = sum(step_ms) if stream_ms is None else stream_ms
    k_ms = sum(a.elapsed_time(b) for a, b in kev) / n_probe
    tmax = torch.tensor([total_ms, statistics.median(step_ms), bracket_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms, median_ms, bracket_ms = float(tmax[0]), float(tmax[1]), float(tmax[2])
    updates_per_step = B * n_total
    value = updates_per_step * args.steps / (total_ms * 1e-3)

    # ---------------- e2e: public API from pinned host batches, losses read back every step ----------------
    e2e_steps = args.steps
    losses_host = torch.zeros(n_local, 3).pin_memory()              # the step's command list ends with the D2H copy into it
    stream = torch.cuda.current_stream()
    for k in range(3):
        ag.update_successor_all(pinned[k % 8], use_gpi=True, host_losses=losses_host)
        stream.synchronize()
    barrier()
    # (a) synchronous: the host waits for every step's losses before it issues the next step (host time fully exposed)
    check = 0.0
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        ag.update_successor_all(pinned[k % 8], use_gpi=True, host_losses=losses_host)
        stream.synchronize()                                        # the step's result is on the host from here on
        check += float(losses_host[0, 0])                           # (read it: D2H of the losses every step)
    barrier()
    assert check == check and check > 0.0, 'e2e losses did not reach the host'
    e2e_sync_s = time.perf_counter() - t0
    # (b) the same loop reading the losses ONE STEP LATE (what a training loop that logs its losses does): step k is issued, then
    # the host waits on the event recorded after step k-1 and reads that step's losses from the other of two pinned buffers.
    # Every step still pulls its batch from pinned host memory and every step's losses are copied back and read inside the
    # timed region; only the host's per-step work overlaps the device's.
    lh = [torch.zeros(n_local, 3).pin_memory() for _ in range(2)]
    evs = [torch.cuda.Event() for _ in range(2)]
    for k in range(2):
        ag.update_successor_all(pinned[k % 8], use_gpi=True, host_losses=lh[k])
    stream.synchronize()
    barrier()
    check = 0.0
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        ag.update_successor_all(pinned[k % 8], use_gpi=True, host_losses=lh[k & 1])
        evs[k & 1].record(stream)
        if k > 0:
            evs[(k - 1) & 1].synchronize()
            check += float(lh[(k - 1) & 1][0, 0])
    evs[(e2e_steps - 1) & 1].synchronize()
    check += float(lh[(e2e_steps - 1) & 1][0, 0])
    barrier()
    assert check == check and check > 0.0, 'e2e (pipelined) losses did not reach the host'
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop()
    e2e_t = torch.tensor([e2e_s, e2e_sync_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_sync_s = float(e2e_t[1])
    e2e_t = e2e_t[0]
    e2e_val = updates_per_step * e2e_steps / float(e2e_t)
    h2d = sum(t.numel() * t.element_size() for t in pinned[0])
    d2h = losses_host.numel() * 4

    # ---------------- in-kernel trace: where the step's time goes without an event between the kernels ----------------
    trace = None
    try:
        if world == 1:
            trace = trace_steps(lambda k: ag.update_successor_all(resident[k % n_res], use_gpi=True))
    except Exception as e:
        trace = {'error': f'{type(e).__name__}: {e}'}

    # ---------------- roofline of the dominant kernel ----------------
    # tensor-core modes: mlp_forward_tc_kernel, ONE launch per step carrying 3 of the step's 5 net passes per (transition,
    # policy): online psi(s), GPI over the library on s' under every task's reward vector, target psi(s').  fp32 mode: the GPI forward.
    # Algorithmic FLOPs (SURVEY 8d): F per (state, policy) pass + 2*A*D per (state, policy, reward vector) for psi . w.
    # Executed FLOPs: what the kernel issues -- K of the input layer padded to 16, psi outputs padded to 16 columns, and the GPI
    # job's output layer in folded form (n_w * A columns, padded) instead of A*D columns followed by the dot with w.
    F = flops_per_net_pass(S, cfg['hidden'], A * D)
    peaks = load_peaks()
    tc_mode = args.precision != 'fp32'
    if tc_mode:
        k_flops = n_local * B * (3 * F + 2 * A * D * n_total)
        wb = 8 if n_total >= 8 else (4 if n_total >= 4 else 1)
        gpi_cols = (((n_total + wb - 1) // wb * wb * A) + 15) // 16 * 16
        hid = 2 * (16 * 256 + 2 * 256 * 256)
        k_exec = n_local * B * (3 * hid + 2 * 2 * 256 * ((A * D + 15) // 16 * 16) + 2 * 256 * gpi_cols)
        kname = ('mlp_forward_tc_kernel: one launch = online psi(s) + fused GPI(s\') + target psi(s\') for all local policies '
                 '(tcgen05 MMA, TMEM accumulators, TMA weight ring)')
    else:
        k_flops = n_local * B * (F + 2 * A * D * n_total)
        k_exec = k_flops
        kname = 'mlp_forward_kernel (GPI form: fused ensemble MLP + GPI epilogue, fp32 CUDA-core mode)'
    achieved = k_flops / (k_ms * 1e-3) / 1e12
    traffic = (load_json('profiles/r02_traffic.json') or {}).get(f'{args.workload}/{args.precision}/n{n_local}')
    roofline = {'kernel': kname, 'bound': 'tensor',
                'achieved': achieved, 'peak': peaks['tf_burst'], 'unit': 'TFLOP/s', 'frac': achieved / peaks['tf_burst'],
                'achieved_executed': k_exec / (k_ms * 1e-3) / 1e12, 'frac_executed': k_exec / (k_ms * 1e-3) / 1e12 / peaks['tf_burst'],
                'traffic': traffic['dram_bytes_per_launch'] if traffic else None,
                'traffic_source': traffic['source'] if traffic else 'no ncu --set full capture of this workload / precision committed',
                'peak_source': f'{peaks["src"]} bf16 cuBLAS burst',
                'kernel_ms': k_ms, 'flops_per_launch': k_flops, 'executed_flops_per_launch': k_exec,
                'in_kernel_window_ms': (trace['forward']['busy_us'] / 1e3) if trace and 'forward' in trace else None,
                'frac_in_kernel_window': (k_flops / (trace['forward']['busy_us'] * 1e-6) / 1e12 / peaks['tf_burst']) if trace and 'forward' in trace else None,
                'timing': 'kernel_ms / achieved / frac: CUDA events recorded by the command list around the kernel inside every timed step '
                          '(mean) -- the bracket includes the launch latency the event exposes (it removes the dependent-launch overlap '
                          'with the prologue kernel); in_kernel_window_ms: the same launch seen from inside (%globaltimer, first CTA past '
                          'its dependency wait -> last CTA exit, isolated steps), see step_trace',
                'note': 'achieved/frac use ALGORITHMIC FLOPs (SURVEY 8d); *_executed count what the kernel issues (folded GPI layer, padded K/N)'}
    step_flops = 5 * F * B * n_local                               # N GPI + N online + N target + 2N backward = 5N passes
    step_tflops = step_flops * args.steps / (total_ms * 1e-3) / 1e12

    # ---------------- M2: GPI action evals/s (BASELINE config 3) ----------------
    gpi_eval = None
    try:
        gpi_eval = {'skipped': '--no-gpi-eval'} if args.no_gpi_eval else time_gpi_eval(world, rank, dev, args.precision, barrier)
    except Exception as e:                                          # the headline line must not depend on the secondary metric
        gpi_eval = {'error': f'{type(e).__name__}: {e}'}

    # ---------------- sharded == unsharded (world > 1) ----------------
    shard = None
    if world > 1:
        try:
            shard = shard_check(cfg, n_local, args.precision, rank, world, dev) if n_total <= 64 else \
                {'skipped': f'{n_total} policies: the unsharded twin is built for <= 64'}
        except Exception as e:
            shard = {'ok': False, 'error': f'{type(e).__name__}: {e}'}
        barrier()

    # ---------------- BASELINE config 4 (ii), strong scaling over this run's GPUs ----------------
    c4s = None
    if world > 1 and not args.no_secondary and not strong:
        try:
            c4s = config4_strong(world, rank, dev, args.precision, barrier)
        except Exception as e:
            c4s = {'error': f'{type(e).__name__}: {e}'}
        barrier()

    out = None
    if rank == 0:
        out = {
            'metric': 'SF TD updates (transitions x tasks)/s', 'value': value, 'unit': 'updates/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': total_ms / args.steps, 'higher_is_better': True,
            'scaling': 'strong' if strong else 'weak', 'vs_baseline': None, 'dtype': 'f32' if args.precision == 'fp32' else args.precision.replace('x3', ''),
            'data': 'synthetic', 'config': workload_config(args.workload, cfg, n_total, world, args.l2),
            'precision_mode': {'name': args.precision, 'what': PRECISION_TEXT[args.precision]},
            'exchange': None if world == 1 else ('peer-memory kernels in the step\'s launch chain (CUDA IPC arenas, signal/wait flags, 128-bit pulls '
                                                 'over NVLink): GPI keys MAX reduce-scatter + [w | delta h] all-gather, no NCCL call inside a step'
                                                 if lib._peer is not None else 'NCCL: all-reduce(MAX) of packed keys + one all-gather'),
            'clocks': clocks,
            'e2e': {'value': e2e_val, 'unit': 'updates/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'ms_per_step': float(e2e_t) / e2e_steps * 1e3,
                    'protocol': 'TSFDQN.update_successor_all(pinned host batch, host_losses=pinned buffer) per step: the prologue kernel pulls the '
                                'batch over PCIe, the Adam launch\'s loss block stores the losses into the pinned host buffer; the host reads every step\'s losses one step late '
                                '(event wait on step k-1 after issuing step k), wall clock around the loop',
                    'sync_value': updates_per_step * e2e_steps / e2e_sync_s, 'sync_ms_per_step': e2e_sync_s / e2e_steps * 1e3,
                    'sync_what': 'the same loop with a stream synchronise + read after EVERY step before the next one is issued'},
            'ms_per_step_median': median_ms,
            'ms_per_step_bracketed': bracket_ms,         # mean of the per-step CUDA-event brackets (each exposes one launch latency)
            'timing': ('value / ms_per_step: the K steps as one stream between two CUDA events (inputs larger than L2); '
                       'ms_per_step_median / _bracketed: an event pair around every step' if args.l2 == 'inputs' else
                       'value / ms_per_step: sum of the per-step CUDA-event brackets, L2 flushed between steps outside the brackets'),
            'warmup_steps_run': n_warm,                     # >= --warmup: a fixed count on every rank, clocks settled under load
            'gpu_launches': launches,
            'roofline': roofline,
            'step_tflops_per_gpu': step_tflops,
            'step_trace': trace,
            'hbm_kernels': hbm_kernels(trace, lib, B, n_local, n_total, peaks) if isinstance(trace, dict) and 'error' not in trace else None,
            'gpi_eval': gpi_eval,
        }
        if shard is not None:
            out['shard_check'] = shard
        if c4s is not None:
            out['config4_strong_scaling'] = c4s
    if world == 1 and rank == 0:
        cores = os.cpu_count() or 1
        timer = Timer(dev)
        with_cpu = not args.no_cpu_baseline
        if with_cpu:
            big = n_total > 8
            cval, cper, kind = cpu_all_task(cfg, n_total, 10 if not big else 1, 2 if not big else 0, cores)
            try:                                                    # SURVEY 8d: "also a 1-thread number" (3 steps)
                c1 = cpu_all_task(cfg, n_total, 3, 1, 1)[0] if not big else None      # (large ensembles: minutes at one thread)
            except Exception:
                c1 = None
            torch.set_num_threads(cores)
            out['cpu_baseline'] = {'value': cval, 'unit': 'updates/s', 'cores': cores, 'kind': kind, 'value_1_thread': c1,
                                   'sample': f'{10 if not big else 1} all-task steps ({n_total} update_successor calls each), B={B}, '
                                             f'{cper * 1e3:.1f} ms/step, ' + ('unmodified reference classes' if kind == 'reference' else 'oracle port') + ' on torch CPU fp32',
                                   'port_vs_reference': load_json('profiles/r02_port_vs_reference.json') if kind == 'port' else None}
        if not args.no_secondary:
            try:
                if args.precision != PARITY_MODE and not strong:
                    pm = measure_steps(cfg, n_local, PARITY_MODE, dev, max(50, min(args.steps, 200)), 20, timer)
                    pm['what'] = PRECISION_TEXT[PARITY_MODE]
                    out['parity_mode'] = pm
                if not strong:
                    out['gpu_eager_baseline'] = gpu_eager_baseline(cfg, n_total, dev)
                    out['configs'] = secondary_configs(args, dev, timer, cores, with_cpu)
            except Exception as e:
                out['secondary_error'] = f'{type(e).__name__}: {e}'
    if rank == 0:
        if args.dump_outputs:
            write_outputs(outputs, args.dump_outputs)
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
