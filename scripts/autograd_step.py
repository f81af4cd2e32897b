"""
Cost of the differentiable psi path on one GPU (prints one JSON object).

(1) One G2 update of one policy at B = 4096, N = 4 (Reacher shapes, hidden 256 x 256) in fp32 and bf16, three ways:
      eager  -- the reference's update body (sfdqn.py:303-371) written in torch on a DeepSF(autograd=True): GPI, psi_model(states),
                target under no_grad, mse losses, backward through PackedSFLibrary.psi, optim.step() (one fused Adam launch)
      fused  -- DeepSF.update_successor (the library's one-command-list train step)
      oracle -- the oracle port (oracle/sf_oracle.py) as eager PyTorch on the GPU (fp32 only: it has no bf16 mode)
(2) The backward pass with a dense dL/dpsi against the train step's sparse one, at B = 4096 for Reacher (N = 4) and Hopper
    (S = 11, A = 27, D = 50, N = 4).  Both timings include the online forward that saves the activations and the split-K
    reduction, so the recorded forward's own time is printed beside them.  The two are not the same work outside the backward
    kernels:
      dense  -- lib.psi(x).backward(d_psi): the forward writes the full psi [B][N][A][D] and allocates its activations (not
                zero-filled), the backward reads an equally large d_psi, allocates a zero-filled gradient of the WHOLE online
                storage [cap][row_stride] and autograd adds it into online.grad;
      sparse -- lib.psi_gradients(x, actions, d_sel): the forward gathers psi(s)[a_b] only, activations and partials live in a
                cached workspace, the result is the reduced [N][row_stride] gradient.
(3) The same two for ONE policy of a 256-policy Hopper library in bf16 (B = 4096): the dense side's gradient and its accumulation
    into online.grad span all 256 rows (about 425 MB each), the cost of making the online storage the autograd leaf.

Times are CUDA-event milliseconds per call (median of --reps windows of --iters calls, after a warm-up); the card's name and power
limit are read in the same run.  Usage: python scripts/autograd_step.py [--iters 50] [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from deep_successor_features_for_transfer_b200.sfdqn import DeepSF  # noqa: E402
from deep_successor_features_for_transfer_b200.workloads import HYPER, ShapeTask, model_lambda  # noqa: E402
from oracle.sf_oracle import OracleSF, synthetic_transitions  # noqa: E402


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ''
    return out or torch.cuda.get_device_name()


def timed(fn, iters, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    res = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        b.synchronize()
        res.append(a.elapsed_time(b) / iters)
    res.sort()
    return round(res[len(res) // 2], 4)


def build(S, A, D, N, precision, autograd, oracle=None):
    sf = DeepSF(pytorch_model_handle=model_lambda([256, 256], ['relu', 'relu']), hyperparameters=dict(HYPER, precision=precision),
                autograd=autograd)
    sf.reset()
    for i in range(N):
        sf.add_training_task(ShapeTask(S, A, D, i))
    if oracle is None:
        return sf
    with torch.no_grad():
        for i in range(N):
            for lin, (W, b) in zip([m for m in sf.psi[i][0][0].net.modules() if isinstance(m, torch.nn.Linear)], oracle.psi[i]):
                lin.weight.data.copy_(W)
                lin.bias.data.copy_(b)
            sf.fit_w[i].weight.data.copy_(oracle.w[i].reshape(1, -1))
    return sf


def eager_update(sf, tr, i):
    """sfdqn.py:303-371 in torch on the packed library (use_gpi=True)."""
    states, actions, rs, phis, next_states, gammas = tr
    (psi_model, _, optim), (target_psi_model, _, _) = sf.psi[i]
    idx = torch.arange(len(gammas), device=states.device)
    with torch.no_grad():
        q1, _ = sf.GPI(next_states, i)
        next_actions = torch.argmax(torch.max(q1, dim=1).values, dim=-1)
        targets = phis + gammas.reshape(-1, 1) * target_psi_model(next_states)[idx, next_actions, :]
    current_psi = psi_model(states)
    merge = current_psi.clone()
    merge[idx, actions, :] = targets
    loss = F.mse_loss(current_psi, merge) + F.mse_loss(sf.fit_w[i](phis), rs)
    optim.zero_grad()
    loss.backward()
    optim.step()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=50)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    gen = torch.Generator().manual_seed(0)
    res = dict(card=card(), unit='ms per call (CUDA events, median of windows)', step={}, backward={})

    S, A, D, N, B, i = 4, 9, 12, 4, 4096, 1
    o = OracleSF(S, A, D, (256, 256), ('relu', 'relu'))
    for _ in range(N):
        o.add_random_policy(gen)
    tr = tuple(v.cuda() for v in synthetic_transitions(B, S, A, D, gen))
    for precision in ('fp32', 'bf16'):
        sf = build(S, A, D, N, precision, True, o)
        eager = timed(lambda: eager_update(sf, tr, i), args.iters, args.reps)
        fused = timed(lambda: sf.update_successor(tr, i, True), args.iters, args.reps)
        res['step'][precision] = dict(eager=eager, fused=fused)
    og = OracleSF(S, A, D, (256, 256), ('relu', 'relu'))
    for W in o.psi:
        og.add_policy([(w.clone(), b.clone()) for w, b in W], o.w[len(og.psi)].clone())
    og.to('cuda')
    res['step']['fp32']['oracle'] = timed(lambda: og.update_successor(tr, i, True), max(1, args.iters // 5), args.reps)

    for name, (S, A, D, hopper) in (('reacher', (4, 9, 12, False)), ('hopper', (11, 27, 50, True))):
        o = OracleSF(S, A, D, (256, 256), ('relu', 'relu'))
        for _ in range(N):
            o.add_random_policy(gen)
        x, actions = (v.cuda() for v in synthetic_transitions(B, S, A, D, gen, hopper=hopper)[:2])
        d_sel = torch.randn(N, B, D, device='cuda') * 1e-4
        d_psi = torch.randn(B, N, A, D, device='cuda') * 1e-4
        for precision in ('fp32', 'bf16', 'tf32x3'):
            lib = build(S, A, D, N, precision, True, o)._library
            res['backward'][f'{name}_{precision}'] = dict(
                recorded_forward=timed(lambda: lib.psi(x, 0, N), args.iters, args.reps),
                forward_plus_sparse_backward=timed(lambda: lib.psi_gradients(x, actions, d_sel, 0, N), args.iters, args.reps),
                forward_plus_dense_backward=timed(lambda: lib.psi(x, 0, N).backward(d_psi), args.iters, args.reps))

    S, A, D, N, i = 11, 27, 50, 256, 7
    lib = build(S, A, D, N, 'bf16', True)._library
    x, actions = (v.cuda() for v in synthetic_transitions(B, S, A, D, gen, hopper=True)[:2])
    d_sel, d_psi = torch.randn(1, B, D, device='cuda') * 1e-4, torch.randn(B, 1, A, D, device='cuda') * 1e-4
    res['backward']['hopper_n256_one_policy_bf16'] = dict(
        online_storage_MB=round(lib.online.numel() * 4 / 2 ** 20, 1),
        recorded_forward=timed(lambda: lib.psi(x, i, 1), args.iters, args.reps),
        forward_plus_sparse_backward=timed(lambda: lib.psi_gradients(x, actions, d_sel, i, 1), args.iters, args.reps),
        forward_plus_dense_backward=timed(lambda: lib.psi(x, i, 1).backward(d_psi), args.iters, args.reps))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
