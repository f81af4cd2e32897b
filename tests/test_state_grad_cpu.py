"""
CPU-only checks of the state-gradient entry point sfgpi_mlp_input_grad: its ctypes struct mirrors include/sfgpi.h, and every
invalid argument is rejected before any CUDA call, with the function's name in the error text.  No call here is valid with a
non-empty batch, so nothing is launched (the pointers are host addresses that are never dereferenced).
"""
import ctypes as C

import pytest

from deep_successor_features_for_transfer_b200 import _lib
from deep_successor_features_for_transfer_b200.library import NetSpec
from tests.test_abi_and_dist_cpu import c_struct_fields

_HOST = (C.c_float * 64)()                           # stands in for device pointers: validation never reads them


def test_input_grad_struct_mirrors_header():
    assert c_struct_fields('sfgpi_input_grad_args') == [f[0] for f in _lib.InputGradArgs._fields_]
    assert 'sfgpi_mlp_input_grad' in _lib.SYMBOLS
    assert _lib.lib().sfgpi_version() == 103


def _args(S=4, precision='bf16', hidden=256, B=64, n_pol=2):
    spec = NetSpec([S, hidden, hidden, hidden, 9 * 12], ['none', 'relu', 'relu', 'none'], 9, 12)
    g = _lib.InputGradArgs()
    g.net, g.precision, g.policy_lo, g.n_pol, g.B = spec.desc(), _lib.PREC[precision], 0, n_pol, B
    g.params = g.dz0 = g.dx = C.addressof(_HOST)
    g.dz0_part_stride = n_pol * B * 256 * 3
    return g


def _rejected(g):
    L = _lib.lib()
    rc = L.sfgpi_mlp_input_grad(C.byref(g) if g is not None else None, None)
    return rc == -1 and b'sfgpi_mlp_input_grad' in L.sfgpi_last_error()


def _with(**kw):
    precision = kw.pop('precision', 'bf16')
    S = kw.pop('S', 4)
    g = _args(S=S, precision=precision)
    for k, v in kw.items():
        setattr(g, k, v)
    return g


@pytest.mark.parametrize('case', [
    dict(params=None), dict(dz0=None), dict(dx=None),
    dict(B=-1), dict(n_pol=-3), dict(policy_lo=-1), dict(dz0_part_stride=-4),
    dict(precision='fp32', B=-1), dict(precision='tf32x3', n_pol=-1),
    dict(S=64, precision='bf16'), dict(S=32, precision='tf32'), dict(S=32, precision='tf32x3'),
    dict(precision='tf32x3', dz0_part_stride=16),     # lo part would overlap hi [n_pol][B][256]
])
def test_input_grad_rejects_invalid_arguments_without_a_gpu(case):
    assert _rejected(_with(**case)), case


def test_input_grad_rejects_unknown_precision_bad_nets_and_null_args():
    assert _rejected(None)
    for prec in (-1, 4, 99):
        g = _args()
        g.precision = prec
        assert _rejected(g) and b'precision' in _lib.lib().sfgpi_last_error()
    g = _args()
    g.net.n_layers = 1                                # no hidden layer: no dZ_0 to read
    assert _rejected(g)
    g = _args(precision='tf32', hidden=128)           # tensor-core modes: hidden width 256 only
    assert _rejected(g)
    g = _args()
    g.net.row_stride = 100                            # W_0 does not fit the row
    assert _rejected(g)


@pytest.mark.parametrize('precision', ['fp32', 'bf16', 'tf32', 'tf32x3'])
def test_input_grad_empty_launch_is_ok(precision):
    """B == 0 or n_pol == 0: rc 0 and nothing launched (no device is needed for that)."""
    L = _lib.lib()
    assert L.sfgpi_mlp_input_grad(C.byref(_args(precision=precision, B=0)), None) == 0
    assert L.sfgpi_mlp_input_grad(C.byref(_args(precision=precision, n_pol=0)), None) == 0
    wide = _args(S=100, precision='fp32', B=0)        # fp32 mode: no S limit
    assert L.sfgpi_mlp_input_grad(C.byref(wide), None) == 0
