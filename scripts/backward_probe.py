"""
A/B timing of the headline train step and its two bf16 backward kernels (prints one JSON object).

Runs `bench.py --gpus 1 --no-cpu-baseline --no-gpi-eval` from each given source tree in turn, --reps rounds alternating the trees
so that both see the same machine state, and keeps from every run:
  value / ms_per_step   the headline (TSFDQN Reacher, B = 4096, 4 policies, bf16, all-task update with GPI), K steps as one stream
  dgrad_us / wgrad_us   the in-kernel busy windows of the two backward kernels (bench.py step_trace: first CTA past its dependency
                        wait -> last CTA exit, median of isolated steps)
  config1 / config5 / config4 / parity_mode   the secondary lines' ms per step (unless --no-secondary)
The card's name and power limit are read in the same run.  Each tree must have been built (__graft_entry__.build()).
Usage: python scripts/backward_probe.py --tree parent=/path/a --tree branch=/path/b [--reps 3] [--steps 200] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys


def card():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return ''


def run_bench(tree, steps, warmup, secondary):
    cmd = [sys.executable, 'bench.py', '--gpus', '1', '--steps', str(steps), '--warmup', str(warmup), '--no-cpu-baseline', '--no-gpi-eval']
    if not secondary:
        cmd.append('--no-secondary')
    r = subprocess.run(cmd, cwd=tree, capture_output=True, text=True)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith('{')]
    if r.returncode != 0 or not lines:
        raise RuntimeError(f'bench.py failed in {tree}:\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}')
    d = json.loads(lines[-1])
    tr = d.get('step_trace') or {}
    out = {'value': d['value'], 'ms_per_step': d['ms_per_step'],
           'dgrad_us': (tr.get('dgrad') or {}).get('busy_us'), 'wgrad_us': (tr.get('wgrad') or {}).get('busy_us'),
           'step_span_us': tr.get('step_span_us')}
    cf = d.get('configs') or {}
    for name, path in (('config1_b32', ('config1_sfdqn_reacher_n4', 'B32', 'gpu')), ('config1_b4096', ('config1_sfdqn_reacher_n4', 'B4096', 'gpu')),
                       ('config5', ('config5_cartpole_b32', 'gpu')), ('config4_all', ('config4_tsfdqn_dissimilar_n256', 'ensemble_all_policies')),
                       ('config4_one', ('config4_tsfdqn_dissimilar_n256', 'sequential_one_policy'))):
        v = cf
        for k in path:
            v = v.get(k) if isinstance(v, dict) else None
        if isinstance(v, list):                                       # one entry per precision: the bf16 one
            v = next((e for e in v if isinstance(e, dict) and e.get('precision') == 'bf16'), None)
        if isinstance(v, dict) and 'ms_per_step' in v:
            out[name] = v['ms_per_step']
    if isinstance(d.get('parity_mode'), dict):
        out['parity_mode'] = d['parity_mode'].get('ms_per_step')
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--tree', action='append', required=True, help='name=path of a built source tree')
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--no-secondary', action='store_true')
    ap.add_argument('--out')
    args = ap.parse_args()
    trees = [t.split('=', 1) for t in args.tree]
    runs = {name: [] for name, _ in trees}
    for _ in range(args.reps):
        for name, path in trees:
            runs[name].append(run_bench(os.path.abspath(path), args.steps, args.warmup, not args.no_secondary))
    summary = {}
    for name, rs in runs.items():
        summary[name] = {k: {'median': statistics.median(v), 'min': min(v), 'max': max(v)}
                         for k in rs[0] if all(r.get(k) is not None for r in rs) for v in [[r[k] for r in rs]]}
    res = {'card': card(), 'reps': args.reps, 'steps': args.steps, 'runs': runs, 'summary': summary,
           'what': 'bench.py --gpus 1 --no-cpu-baseline --no-gpi-eval per tree, trees alternated; ms are per step, us are in-kernel '
                   'busy windows (step_trace)'}
    text = json.dumps(res)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')
    print(text)


if __name__ == '__main__':
    main()
