"""
-m gpu: the two modes of the bf16 dgrad kernel agree, and so do the weight gradients stored from them.  A backward of <= 148
row tiles runs mlp_dgrad_tc_kernel in one-tile mode (one tile per CTA, 8-stage weight ring), a larger one in paired mode (two
tiles ping-pong); both issue the same MMA sequence into each accumulator, so dz / dzo are equal bit for bit.  An 8-policy
library whose first 4 nets are the 4-policy library's nets runs paired at B = 4096 (256 tiles) where the 4-policy one runs one
tile per CTA (128 tiles).  The weight gradients come from the same kernel in both (fp32 tiles written to grad_part by bulk
tensor stores); they are equal bit for bit where the split-K counts agree, otherwise within fp32 reduction-order tolerance.
"""
import pytest
import torch

from oracle.sf_oracle import OracleSF, synthetic_transitions
from tests import gpu_util as gu

pytestmark = pytest.mark.gpu
HYPER_BF16 = dict(gu.HYPER, precision='bf16')


def _lib(S, A, D, acts, N, seed):
    gen = torch.Generator().manual_seed(seed)                      # same seed: the first nets of every N are the same nets
    o = OracleSF(S, A, D, (256, 256), tuple(acts))
    for _ in range(N):
        o.add_random_policy(gen)
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=list(acts), N=N)
    return gu.build_g2(meta, oracle=o, hyper=HYPER_BF16)._library


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


@pytest.mark.parametrize('dense', [False, True])
@pytest.mark.parametrize('S,A,D,acts,B', [
    (4, 9, 12, ('relu', 'relu'), 4096),   # Reacher headline shape: 128 vs 256 tiles
    (4, 9, 12, ('relu', 'relu'), 4000),   # ragged last tile
    (4, 9, 12, ('relu', 'relu'), 32),     # one partial tile per policy (both launches one tile per CTA)
    (4, 2, 20, ('tanh', 'tanh'), 4096),   # tanh CartPole net: the epilogue reads the saved activations
])
def test_one_tile_and_paired_backward_agree(S, A, D, acts, B, dense):
    small, large = _lib(S, A, D, acts, 4, seed=5), _lib(S, A, D, acts, 8, seed=5)
    gen = torch.Generator().manual_seed(9)
    x, actions = (v.cuda() for v in synthetic_transitions(B, S, A, D, gen)[:2])
    d8 = (torch.randn(8, B, D, generator=gen) * 1e-3).cuda()
    grads, ws = [], []
    for lib, n_pol in ((small, 4), (large, 8)):
        if dense:
            g = torch.zeros(B, n_pol, A, D, device='cuda')
            g[torch.arange(B, device='cuda'), :, actions, :] = d8[:n_pol].transpose(0, 1)
            g += (torch.randn(B, n_pol, A, D, generator=gen) * 1e-4).cuda()          # dense: every psi entry has a gradient
            if n_pol == 8:
                g[:, :4] = g4                                                      # the shared nets get the same dL/dpsi
            g4 = g[:, :4].clone()
            _, acts_, masks = lib._psi_forward(x, 0, n_pol)
            grad, _ = lib._psi_backward(x, 0, n_pol, acts_, masks, g)
            grads.append(grad[:n_pol])
        else:
            grads.append(lib.psi_gradients(x, actions, d8[:n_pol], 0, n_pol))
        torch.cuda.synchronize()
        ws.append(lib._ws[(B, n_pol)])
    assert torch.equal(ws[0]['dzo'], ws[1]['dzo'][:4])
    assert torch.equal(ws[0]['dz'], ws[1]['dz'][:, :4])
    got, ref = grads[0][:4], grads[1][:4]
    if ws[0]['n_split'] == ws[1]['n_split']:
        assert torch.equal(got, ref)
    else:
        for p in range(4):
            assert _rel(got[p], ref[p]) < 1e-5, f'policy {p}: {_rel(got[p], ref[p])}'
