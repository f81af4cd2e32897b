"""Per-layer relative Frobenius errors of the tf32 / tf32x3 backward kernels against fp32 autograd (developer probe)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from tests import test_gpu_tf32 as tt
from tests import gpu_util as gu
from oracle.sf_oracle import synthetic_transitions

for precision in sys.argv[1:] or ['tf32x3']:
    for (S, A, D, N, B, hopper) in [(4, 9, 12, 2, 128, False), (4, 9, 12, 2, 256, False), (4, 9, 12, 3, 1000, False), (11, 27, 50, 2, 300, True), (4, 2, 20, 2, 32, False)]:
        meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
        o, gen = tt.make_oracle(S, A, D, N, seed=77)
        sf = gu.build_g2(meta, oracle=o, hyper=dict(gu.HYPER, precision=precision))
        lib = sf._library
        tr = synthetic_transitions(B, S, A, D, gen, hopper=hopper)
        x, actions = tr[0], tr[1]
        lo, n_pol = (1, N - 1)
        d_out = torch.randn(n_pol, B, D, generator=gen) * 1e-4
        ref = tt.torch_psi_grads(o, lo, n_pol, x, actions, d_out)
        got = lib.psi_gradients(x.cuda(), actions.cuda(), d_out.cuda(), lo, n_pol).cpu()
        ws = lib._workspace(B, n_pol)
        errs = []
        for p in range(n_pol):
            for l, ((W, b), (gW, gb)) in enumerate(zip(lib.spec.views(got[p]), ref[p])):
                errs.append(f'p{p}L{l}: dW {tt.fro_err(W, gW):.2e} db {tt.fro_err(b, gb):.2e}')
        print(precision, (S, A, D, N, B), 'n_split', ws['n_split'], ' | '.join(errs), flush=True)
