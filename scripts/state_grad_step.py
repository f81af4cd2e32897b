"""
Cost of the state gradient of the packed psi networks on one GPU (prints one JSON object).

At B = 4096, N = 4 (hidden 256 x 256), for Reacher (S = 4, A = 9, D = 12) and Hopper (S = 11, A = 27, D = 50) in all four precision
modes:
  without        lib.psi(x).backward(d_psi) on states that do not require grad: forward + dense backward (scripts/autograd_step.py)
  with           the same on states that require grad (library built with state_grad=True): + one sfgpi_mlp_input_grad launch,
                 the dx allocation and its accumulation into x.grad.  The two alternate window by window in the same run.
  kernel_us      sfgpi_mlp_input_grad alone, back to back (the launches are queued behind a sleep kernel, so the host is not timed):
                 l2_warm = dZ0 read again right after the previous call, as in the backward (it was just written there);
                 l2_flushed = a 256 MB write between calls evicts dZ0 from the 126 MB L2, timed per call.
  bytes          dZ0 (n_pol*B*256 elements: bf16, fp32, fp32 hi + lo) + W0 (n_pol*256*S fp32) + dx (B*S fp32), and bytes / kernel time
                 against the HBM bandwidth of MEASURED_PEAKS.json (the figure DESIGN.md quotes when that file is absent).

Times are CUDA-event milliseconds per call (median of --reps windows of --iters calls, after a warm-up); the card's name and power
limit are read in the same run.  Usage: python scripts/state_grad_step.py [--iters 50] [--reps 7] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from deep_successor_features_for_transfer_b200 import _lib  # noqa: E402
from deep_successor_features_for_transfer_b200.library import _stream  # noqa: E402
from deep_successor_features_for_transfer_b200.sfdqn import DeepSF  # noqa: E402
from deep_successor_features_for_transfer_b200.workloads import HYPER, ShapeTask, model_lambda  # noqa: E402
from oracle.sf_oracle import OracleSF, synthetic_transitions  # noqa: E402
from scripts.autograd_step import card  # noqa: E402

HBM_GBPS_DESIGN = 6547.0          # DESIGN.md section 5: the measured copy bandwidth recorded in MEASURED_PEAKS.json


def build(S, A, D, N, precision, oracle):
    sf = DeepSF(pytorch_model_handle=model_lambda([256, 256], ['relu', 'relu']), hyperparameters=dict(HYPER, precision=precision),
                autograd=True, state_grad=True)
    sf.reset()
    for i in range(N):
        sf.add_training_task(ShapeTask(S, A, D, i))
    with torch.no_grad():
        for i in range(N):
            for lin, (W, b) in zip([m for m in sf.psi[i][0][0].net.modules() if isinstance(m, torch.nn.Linear)], oracle.psi[i]):
                lin.weight.data.copy_(W)
                lin.bias.data.copy_(b)
    return sf._library


def hbm_peak():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'MEASURED_PEAKS.json'
    except (OSError, KeyError, ValueError):
        return HBM_GBPS_DESIGN, 'DESIGN.md (MEASURED_PEAKS.json not present)'


def timed_pair(fa, fb, iters, reps):
    """Median ms per call of fa and fb, their windows alternating."""
    for _ in range(3):
        fa()
        fb()
    torch.cuda.synchronize()
    res = ([], [])
    for _ in range(reps):
        for k, fn in enumerate((fa, fb)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                fn()
            b.record()
            b.synchronize()
            res[k].append(a.elapsed_time(b) / iters)
    return [round(sorted(r)[len(r) // 2], 4) for r in res]


def kernel_times(launch, iters, reps):
    """(l2_warm, l2_flushed) microseconds per sfgpi_mlp_input_grad launch."""
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device='cuda')
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    warm = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(50_000_000)                      # the GPU waits while the host queues the launches
        a.record()
        for _ in range(iters):
            launch()
        b.record()
        b.synchronize()
        warm.append(a.elapsed_time(b) * 1e3 / iters)
    cold = []
    for _ in range(reps):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        torch.cuda._sleep(50_000_000)
        for a, b in ev:
            flush.fill_(1)
            a.record()
            launch()
            b.record()
        torch.cuda.synchronize()
        cold.extend(a.elapsed_time(b) * 1e3 for a, b in ev)
    return round(sorted(warm)[len(warm) // 2], 2), round(sorted(cold)[len(cold) // 2], 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=50)
    ap.add_argument('--reps', type=int, default=7)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    gen = torch.Generator().manual_seed(0)
    peak, peak_src = hbm_peak()
    res = dict(card=card(), unit='ms per call (CUDA events, median of windows); kernel_us in microseconds', hbm_peak_GBps=peak,
               hbm_peak_source=peak_src, B=4096, N=4, runs={})
    N, B = 4, 4096
    for name, (S, A, D, hopper) in (('reacher', (4, 9, 12, False)), ('hopper', (11, 27, 50, True))):
        o = OracleSF(S, A, D, (256, 256), ('relu', 'relu'))
        for _ in range(N):
            o.add_random_policy(gen)
        x = synthetic_transitions(B, S, A, D, gen, hopper=hopper)[0].cuda()
        d_psi = torch.randn(B, N, A, D, device='cuda') * 1e-4
        for precision in ('fp32', 'bf16', 'tf32', 'tf32x3'):
            lib = build(S, A, D, N, precision, o)
            xr = x.clone().requires_grad_(True)

            def with_dx():
                xr.grad = None
                lib.psi(xr, 0, N).backward(d_psi)
            without, with_ = timed_pair(lambda: lib.psi(x, 0, N).backward(d_psi), with_dx, args.iters, args.reps)
            ws = lib._workspace(B, N)                          # holds the last backward's dZ0
            dx = lib._input_grad(ws, 0, N, B)
            assert torch.equal(dx, xr.grad)
            g = ws['input_grad']                                  # the launch _input_grad makes, without its Python around it
            fn, st = _lib.lib().sfgpi_mlp_input_grad, _stream()
            assert fn(C.byref(g), st) == 0, _lib.lib().sfgpi_last_error()
            warm, cold = kernel_times(lambda: fn(C.byref(g), st), args.iters, args.reps)
            elem = {'bf16': 2, 'fp32': 4, 'tf32': 4, 'tf32x3': 8}[precision]
            nbytes = N * B * 256 * elem + N * 256 * S * 4 + B * S * 4
            res['runs'][f'{name}_{precision}'] = dict(
                forward_plus_dense_backward=without, with_state_grad=with_, added_pct=round(100 * (with_ - without) / without, 1),
                kernel_us=dict(l2_warm=warm, l2_flushed=cold), bytes=nbytes,
                GBps=dict(l2_warm=round(nbytes / warm / 1e3, 1), l2_flushed=round(nbytes / cold / 1e3, 1)),
                hbm_fraction_l2_flushed=round(nbytes / cold / 1e3 / peak, 3))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
