"""
-m gpu: sfgpi_adam_step called directly.  Every per-optimizer segment of a launch is stepped either in a 128-bit range (4
parameters per thread: length, strides and pointers all 16-byte aligned) or in a scalar range (1 per thread).  The per-element
arithmetic is the same in both, so stepping the same values from aligned storage and from storage one float off must give the
same bits -- fresh and clamped segments included, and whatever mix of range kinds and shared segments a launch holds.  One
call also advances `step` and writes the next step's bias corrections into `consts_next`, and a fresh call touches neither.
"""
import ctypes as C
import math

import pytest
import torch

from deep_successor_features_for_transfer_b200 import _lib
from deep_successor_features_for_transfer_b200.library import AdamSeg, NetSpec, _stream, adam_args

pytestmark = pytest.mark.gpu

ROW = NetSpec([4, 256, 256, 256, 108], ['none', 'relu', 'relu', 'none'], 9, 12).row_stride      # a psi row (Reacher)


def _data(specs, n_pol, seed):
    """Host values of every segment: parameters (one row if shared), moments and gradient partials, rows padded to 4 floats."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for sp in specs:
        st = (sp['len'] + 3) // 4 * 4
        out.append(dict(p=torch.randn(1 if sp.get('shared') else n_pol, st, generator=g),
                        m=0.1 * torch.randn(n_pol, st, generator=g), v=0.01 * torch.rand(n_pol, st, generator=g),
                        g=torch.randn(n_pol, sp['n_part'], st, generator=g)))
    return out


def _place(t, shift):
    """t on the device, its first element `shift` floats past a 16-byte boundary."""
    buf = torch.zeros(t.numel() + 4, dtype=torch.float32, device='cuda')
    view = buf[shift:shift + t.numel()].view(t.shape)
    view.copy_(t)
    return view


def _step(specs, data, n_pol, shifts, step0=None, null_mv=False):
    """
    One sfgpi_adam_step over the segments placed at `shifts`; step0 None: a fresh launch, null_mv: without moment buffers.
    -> [p, m, v] of every segment, step, consts, consts_next (device tensors after the call), consts as it was passed.
    """
    segs, bufs, grads = [], [], []                                    # (grads: alive until the launch has run)
    for sp, d, sh in zip(specs, data, shifts):
        p, m, v, g = (_place(d[k], sh) for k in 'pmvg')
        st = p.shape[1]
        segs.append(AdamSeg(p.data_ptr(), None if null_mv else m.data_ptr(), None if null_mv else v.data_ptr(), g.data_ptr(), sp['len'],
                            sp.get('lr', 1e-3), sp.get('wd', 0.0), param_stride=0 if sp.get('shared') else st, mv_stride=st,
                            grad_pol_stride=sp['n_part'] * st, grad_part_stride=st, n_part=sp['n_part'], clamp=sp.get('clamp')))
        bufs += [p, m, v]
        grads.append(g)
    step = torch.zeros(n_pol, dtype=torch.int32) if step0 is None else step0
    t = step.double() + 1
    consts = torch.stack([1.0 - 0.9 ** t, torch.sqrt(1.0 - 0.999 ** t)], dim=1).cuda()
    step, consts_next, consts0 = step.cuda(), torch.zeros_like(consts), consts.clone()
    ad = adam_args(segs, n_pol, None if step0 is None else step.data_ptr(), (consts.data_ptr(), consts_next.data_ptr()))
    _lib.call('sfgpi_adam_step', C.byref(ad), _stream())
    torch.cuda.synchronize()
    return bufs + [step, consts, consts_next, consts0]


def _same_bits(specs, n_pol, shifts, fresh=False, seed=0):
    data = _data(specs, n_pol, seed)
    step0 = None if fresh else torch.randint(0, 7, (n_pol,), generator=torch.Generator().manual_seed(seed), dtype=torch.int32)
    a = _step(specs, data, n_pol, shifts, step0)
    b = _step(specs, data, n_pol, [1] * len(specs), step0, null_mv=fresh)      # every segment one float off 16 bytes: scalar ranges
    for k, (x, y) in enumerate(zip(a, b)):
        if not (fresh and k % 3 and k < 3 * len(specs)):                 # (fresh: b has no moment buffers)
            assert torch.equal(x, y), k
    if fresh:                                                            # moments start at 0: neither read nor stored
        for k, d in enumerate(data):
            assert torch.equal(a[3 * k + 1].cpu(), d['m']) and torch.equal(a[3 * k + 2].cpu(), d['v'])
    for k, d in enumerate(data):                                          # the step moved every parameter
        assert not torch.equal(a[3 * k][:, :specs[k]['len']].cpu(), d['p'][:, :specs[k]['len']])


@pytest.mark.parametrize('n_part', [1, 2, 5])
@pytest.mark.parametrize('wd', [0.0, 1e-2])
def test_128bit_and_scalar_ranges_agree(n_part, wd):
    specs = [dict(len=n, n_part=n_part, wd=wd, lr=lr) for n, lr in ((1, 1e-3), (3, 3e-4), (4, 1e-3), (5, 1e-2), (1027, 1e-3),
                                                                    (ROW, 5e-4))]
    _same_bits(specs, 2, [0] * len(specs), seed=n_part)


def test_clamped_segments_agree():
    specs = [dict(len=4, n_part=1, clamp=(-0.5, 0.5), lr=0.3), dict(len=1024, n_part=2, wd=1e-2, clamp=(-0.2, 0.3), lr=0.3),
             dict(len=1027, n_part=1, clamp=(0.0, 1e6), lr=0.3)]
    _same_bits(specs, 2, [0, 0, 0], seed=3)


def test_fresh_launch_agrees():
    specs = [dict(len=ROW, n_part=3), dict(len=12, n_part=1), dict(len=1, n_part=1), dict(len=1, n_part=1, clamp=(1e-2, 1e6))]
    _same_bits(specs, 1, [0, 0, 0, 0], fresh=True, seed=4)


def test_mixed_ranges_and_shared_segment_in_one_launch():
    """3 optimizers: an aligned own segment (128-bit), an unaligned one (scalar) and a tensor they share, in one launch."""
    specs = [dict(len=1024, n_part=2, wd=1e-2), dict(len=1024, n_part=2, lr=3e-4), dict(len=300, n_part=1, shared=True, lr=1e-2)]
    _same_bits(specs, 3, [0, 1, 0], seed=5)


def test_step_and_bias_corrections_advance_in_the_launch():
    specs = [dict(len=1024, n_part=1), dict(len=5, n_part=1)]
    data = _data(specs, 3, 6)
    step0 = torch.tensor([0, 4, 9], dtype=torch.int32)
    *_, step, consts, consts_next, consts0 = _step(specs, data, 3, [0, 0], step0)
    assert torch.equal(step.cpu(), step0 + 1) and torch.equal(consts, consts0)                  # consts: read only
    want = torch.tensor([[1.0 - 0.9 ** (s + 2), math.sqrt(1.0 - 0.999 ** (s + 2))] for s in step0.tolist()], dtype=torch.float64)
    assert torch.allclose(consts_next.cpu(), want, rtol=1e-13, atol=0.0)
    *_, step, consts, consts_next, consts0 = _step(specs, data, 3, [0, 0])             # fresh: none of the three is touched
    assert torch.equal(step.cpu(), torch.zeros(3, dtype=torch.int32)) and torch.equal(consts, consts0) and not consts_next.any()
