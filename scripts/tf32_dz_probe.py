"""Which rows of the stored dZ / activations differ from autograd (developer probe for the tf32x3 backward)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from tests import test_gpu_tf32 as tt
from tests import gpu_util as gu
from oracle.sf_oracle import synthetic_transitions, act_fn

S, A, D, N, B = 4, 9, 12, 3, int(sys.argv[1]) if len(sys.argv) > 1 else 1000
meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
o, gen = tt.make_oracle(S, A, D, N, seed=77)
sf = gu.build_g2(meta, oracle=o, hyper=dict(gu.HYPER, precision='tf32x3'))
lib = sf._library
tr = synthetic_transitions(B, S, A, D, gen)
x, actions = tr[0], tr[1]
lo, n_pol = 1, N - 1
d_out = torch.randn(n_pol, B, D, generator=gen) * 1e-4
got = lib.psi_gradients(x.cuda(), actions.cuda(), d_out.cuda(), lo, n_pol).cpu()
ws = lib._workspace(B, n_pol)
acts = ws['acts'].sum(0).cpu()      # [L-1][n_pol][B][256]
dz = ws['dz'].sum(0).cpu()
dzo = ws['dzo'].sum(0).cpu()
for p in range(n_pol):
    layers = o.psi[lo + p]
    hs, zs = [], []
    h = x
    for (W, b), a in zip(layers, o.acts):
        z = torch.addmm(b, h, W.t())
        h = act_fn(a)(z)
        hs.append(h); zs.append(z)
    # reference dZ chain
    dzL = torch.zeros(B, A * D)
    for b_ in range(B):
        dzL[b_, actions[b_] * D:(actions[b_] + 1) * D] = d_out[p, b_]
    dzs = {3: dzL}
    for l in (2, 1, 0):
        dA = dzs[l + 1] @ layers[l + 1][0]
        dzs[l] = dA * ((zs[l] > 0).float() if o.acts[l] == 'relu' else 1.0)
    for l in range(3):
        ea = (acts[l, p] - hs[l]).abs().max(dim=1).values / hs[l].abs().max()
        ed = (dz[l, p] - dzs[l]).abs().max(dim=1).values / dzs[l].abs().max()
        bad_a = (ea > 1e-5).nonzero().flatten().tolist()
        bad_d = (ed > 1e-4).nonzero().flatten().tolist()
        print(f'pl{p} layer{l}: acts max err {float(ea.max()):.2e} bad rows {bad_a[:12]} ({len(bad_a)}) | dz max err {float(ed.max()):.2e} bad rows {bad_d[:12]} ({len(bad_d)})')
    ez = (dzo[p][:, :A * D] - dzL).abs().max()
    print(f'pl{p} dzo err {float(ez):.2e}')
