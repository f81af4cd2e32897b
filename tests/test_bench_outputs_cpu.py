"""CPU: bench.py --dump-outputs writes every array whole while they fit its byte cap, a fixed seeded sample of the largest otherwise."""
import numpy as np

import bench


def test_dump_outputs_whole_when_they_fit(tmp_path):
    arrays = {'losses': np.arange(12, dtype=np.float32).reshape(4, 3), 'h': np.linspace(-1, 1, 1212, dtype=np.float32)}
    bench.write_outputs(arrays, str(tmp_path / 'out'))
    for k, a in arrays.items():
        got = np.load(tmp_path / 'out' / f'{k}.npy')
        assert got.dtype == np.float32 and got.shape == a.shape and np.array_equal(got, a)


def test_dump_outputs_sample_the_largest_array_down_to_the_cap(tmp_path):
    arrays = {'losses': np.full((4, 3), 0.5, dtype=np.float32), 'psi_online': np.arange(50_000, dtype=np.float32)}
    cap = 40_000
    for d in ('a', 'b'):
        bench.write_outputs(arrays, str(tmp_path / d), max_bytes=cap)
    losses, psi = np.load(tmp_path / 'a' / 'losses.npy'), np.load(tmp_path / 'a' / 'psi_online.npy')
    assert np.array_equal(losses, arrays['losses'])                          # small arrays stay whole
    assert losses.nbytes + psi.nbytes <= cap and psi.size > 0.9 * (cap - losses.nbytes) / 4
    assert psi.dtype == np.float32 and np.all(np.diff(psi) > 0) and psi[-1] < 50_000      # distinct elements, in index order
    assert np.array_equal(psi, np.load(tmp_path / 'b' / 'psi_online.npy'))   # the same sample every run
