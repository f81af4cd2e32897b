"""
The TD step (csrc/td.cu, sfgpi_td_step) and the two other loss heads that feed Adam partials (sfgpi_phi_head, sfgpi_g4_head),
output by output against a float64 autograd restatement of the reference's loss.  The rest of the suite sees these kernels only
through post-Adam weights, and Adam hides most gradient errors: its first step is about lr * sign(g), and a constant positive
factor on a gradient cancels at every step.  So the outputs themselves are checked here -- d_out (which seeds the psi backward),
the loss partials and the gradient row of w, g (its Linear and its planar flows) and h -- at the batch sizes where the CTA /
cluster partitioning has edges, in every variant, with both forms of the next value, at several TSF shapes and across the
shared-memory sizes where the launch needs an opt-in.

Tolerance: every output within 1e-5 of the float64 reference's max-abs value (gradient rows: per parameter block).  fp32
summation over a few thousand rows stays well inside that; a dropped tail row at B = 257 moves dw by about 4e-3 of its
scale, a dropped partial or a wrong constant by O(1).

Only test_td_reference_matches_oracle runs without a GPU: it pins the float64 reference to the CPU oracle.
"""
import ctypes as C

import pytest
import torch

from oracle.sf_oracle import OracleSF, g_apply, init_linear, mlp_forward, synthetic_transitions
from deep_successor_features_for_transfer_b200 import _lib

TOL = 1e-5
E_INVALID, E_SMEM = -1, -2
SENTINEL = 1234.5                  # value of the tails behind every output: a kernel must never write there
TAIL = 64
KMAX_SMEM = 227 * 1024             # csrc/common.cuh kMaxSmem: the B200's per-block opt-in limit
TD_STATIC_SMEM = 32 * 4            # td_kernel: __shared__ int astar_s[32]
ADAPT_STATIC_SMEM = 8 * 4          # target_adapt_kernel: __shared__ float red[8]
F = torch.nn.functional


# ---- the float64 reference ------------------------------------------------------------------------------------------------------
def split_g(g_row, S, G, K):
    """Packed g row W[G][S] | b[G] | K x (weight[S] | bias | scale[S]) -> the oracle's g form (g_apply)."""
    lin = (g_row[:G * S].view(G, S), g_row[G * S:G * S + G])
    if K == 0:
        return lin
    flows = []
    for k in range(K):
        o = G * S + G + k * (2 * S + 1)
        flows.append((g_row[o:o + S].view(1, S), g_row[o + S:o + S + 1], g_row[o + S + 1:o + 2 * S + 1].view(1, S)))
    return flows + [lin]


def td_reference(variant, cur, nxt, phis, rs, gammas, w, A, beta=1.0, g_row=None, h=None, s=None, s1=None, G=0, K=0):
    """
    One policy's TD loss in float64, as OracleSF.update_successor (variants 0, 1) and tsf_update_successor (variant 2) compute it,
    on inputs already gathered: cur = psi(s)[a] [B][D], nxt = psi^-(s')[a*] [B][D]; g_row is the packed g row, h = Wh | bh.
        l1 = sum diff^2 / (B A D)      l2 = sum e^2 / B      loss = l1 (variant 0) or l1 + beta l2
    In variant 2 phi~ = phi * (h(g(s)) + h(g(s'))) and the targets carry gradient into g and h.  Returns (sum diff^2, sum e^2,
    dL/dcur [B][D], gradient row) with the row in sfgpi_td_step's layout [dw | dWg | dbg | flows | dWh | dbh] (variant 1: dw,
    variant 0: empty).
    """
    f = lambda x: torch.as_tensor(x).detach().cpu().double()
    cur = f(cur).requires_grad_(True)
    B, D = cur.shape
    phis, gm = f(phis), f(gammas).reshape(-1, 1)
    leaves, tphis = [cur], phis
    if variant >= 1:
        w_leaf = f(w).reshape(1, D).requires_grad_(True)
        leaves.append(w_leaf)
    if variant == 2:
        S = s.shape[1]
        g_leaf, h_leaf = f(g_row).requires_grad_(True), f(h).requires_grad_(True)
        g_fn = split_g(g_leaf, S, G, K)
        Wh, bh = h_leaf[:D * G].view(D, G), h_leaf[D * G:]
        aff = F.linear(g_apply(f(s), g_fn), Wh, bh) + F.linear(g_apply(f(s1), g_fn), Wh, bh)
        tphis = aff * phis
        leaves += [g_leaf, h_leaf]
    diff = cur - (tphis + gm * f(nxt))
    l1s = (diff ** 2).sum()
    loss, l2s = l1s / (B * A * D), torch.zeros((), dtype=torch.float64)
    if variant >= 1:
        e = F.linear(tphis, w_leaf).reshape(-1) - f(rs).reshape(-1)
        l2s = (e ** 2).sum()
        loss = loss + beta * l2s / B
    grads = torch.autograd.grad(loss, leaves)
    row = torch.cat([gr.reshape(-1) for gr in grads[1:]]) if variant else torch.zeros(0, dtype=torch.float64)
    return float(l1s.detach()), float(l2s.detach()), grads[0], row


def row_blocks(variant, D, S=0, G=0, K=0):
    """Lengths of the parameter blocks of a gradient row (each is compared against its own scale)."""
    if variant == 0:
        return []
    if variant == 1:
        return [D]
    return [n for n in (D, G * S, G, K * (2 * S + 1), D * G, D) if n]


def err(got, ref):
    got, ref = torch.as_tensor(got).detach().cpu().double(), torch.as_tensor(ref).detach().cpu().double()
    assert got.shape == ref.shape, (got.shape, ref.shape)
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)) if ref.numel() else 0.0


def assert_row_close(got, ref, blocks, what, tol=TOL):
    assert got.numel() == ref.numel() == sum(blocks)
    o = 0
    for k, n in enumerate(blocks):
        e = err(got.reshape(-1)[o:o + n], ref.reshape(-1)[o:o + n])
        assert e < tol, f'{what}: gradient block {k} (floats {o}..{o + n}) off by {e:.3g} of its scale'
        o += n


def g_row_of(g):
    """The oracle's g (Linear, or flows + Linear) -> packed row W | b | K x (weight | bias | scale)."""
    if isinstance(g, tuple):
        return torch.cat([g[0].reshape(-1), g[1].reshape(-1)])
    W, b = g[-1]
    return torch.cat([W.reshape(-1), b.reshape(-1)] + [t.reshape(-1) for fl in g[:-1] for t in fl])


@pytest.mark.parametrize('variant,K', [(0, 0), (1, 0), (2, 0), (2, 2)])
def test_td_reference_matches_oracle(variant, K):
    """The float64 reference against the oracle's own step: losses, last_grads of w, g, h, and of psi via dL/dcur."""
    S, A, D, G, B, N, i = 3, 4, 5, 6, 37, 2, 1
    beta = 2.5 if variant == 2 else 1.0
    gen = torch.Generator().manual_seed(100 + 10 * variant + K)
    o = OracleSF(S, A, D, hidden=(16, 16), tsf_dim=G if variant == 2 else None, beta=beta)
    for _ in range(N):
        layers = [init_linear(o.dims[l + 1], o.dims[l], gen) for l in range(len(o.dims) - 1)]
        g = h = None
        if variant == 2:
            g = init_linear(G, S, gen)
            if K:
                g = [tuple(torch.randn(*sh, generator=gen) * 0.5 for sh in ((1, S), (1,), (1, S))) for _ in range(K)] + [g]
            h = init_linear(D, G, gen)
        o.add_policy(layers, torch.rand(1, D, generator=gen) - 0.5, g, h)
    tr = synthetic_transitions(B, S, A, D, gen)
    states, actions, rs, phis, next_states, gammas = tr
    idx = torch.arange(B)
    layers0 = [(W.clone(), b.clone()) for W, b in o.psi[i]]
    with torch.no_grad():
        nxt = o.get_next_successor(next_states, i)[idx, o.next_actions(next_states, i, True)]
        cur = o.get_successor(states, i)[idx, actions]
    w0 = o.w[i].clone()
    g0 = g_row_of(o.g[i]) if variant == 2 else None
    h0 = torch.cat([o.h[0].reshape(-1), o.h[1]]) if variant == 2 else None
    if variant == 2:
        out = o.tsf_update_successor(tr, i, True)
    elif variant == 1:
        out = o.update_successor(tr, i, True)
    else:
        out = o.update_successor((states, actions, phis, next_states, gammas), i, True, with_reward_loss=False)
    l1s, l2s, dcur, row = td_reference(variant, cur, nxt, phis, rs, gammas, w0, A, beta, g0, h0, states, next_states, G, K)
    l1, l2 = l1s / (B * A * D), l2s / B
    assert abs(float(out[1]) - l1) <= TOL * l1 and abs(float(out[2]) - l2) <= TOL * max(l2, 1e-30)
    assert abs(float(out[0]) - (l1 + beta * l2 if variant else l1)) <= TOL * float(out[0])
    lg = o.last_grads
    parts = []
    if variant >= 1:
        parts.append(lg['w'][0].reshape(-1))
    if variant == 2:
        gg = lg['g']                                               # g_flat order: flows (weight, bias, scale)..., then W, b
        parts += [gg[-2].reshape(-1), gg[-1].reshape(-1)] + [t.reshape(-1) for t in gg[:-2]]
        parts += [t.reshape(-1) for t in lg['h']]
    if parts:
        assert_row_close(torch.cat(parts), row, row_blocks(variant, D, S, G, K), 'oracle')
    # dL/dcur, pushed back through psi, is the oracle's psi gradient
    leaves = [t.clone().requires_grad_(True) for Wb in layers0 for t in Wb]
    psi = mlp_forward([(leaves[2 * l], leaves[2 * l + 1]) for l in range(len(layers0))], o.acts, states).reshape(B, A, D)
    for got, ref in zip(torch.autograd.grad(psi[idx, actions], leaves, grad_outputs=dcur.float()), lg['sf']):
        assert err(got, ref) < TOL


# ---- direct calls of sfgpi_td_step ----------------------------------------------------------------------------------------------
def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def guarded(n, poison=float('nan')):
    """Device buffer of n floats (set to `poison`) followed by a sentinel tail; returns (whole buffer, view of the n floats)."""
    buf = torch.full((n + TAIL,), SENTINEL, dtype=torch.float32, device='cuda')
    buf[:n] = poison
    return buf, buf[:n]


def td_smem_bytes(variant, D, S=0, G=0, K=0, own_mc=True):
    """Dynamic shared memory of one TD launch: the host code's byte formula (csrc/td.cu, sfgpi_td_step) restated."""
    tsf = variant == 2
    n_red = D + D * S + D + K * (2 * S + 1) if tsf else D
    fl = D + 4 * 32 * D + 3 * 32 + 8 + n_red + 2
    if tsf:
        fl += D * S + D + 2 * 32 * S + (G * S + G + D * G + D if own_mc else 0)
    if K > 0:
        fl += 3 * K * (2 * S + 1) + 2 * 32 * ((K + 1) * S + K)
    return 4 * fl


def make_td_case(variant, B, n_pol, S=4, A=9, D=12, G=100, K=0, next_form='sel', seed=0):
    """Seeded inputs of one TD launch (CPU fp32).  w and g rows carry padding (w_stride, g_stride larger than the data) filled
    with finite garbage; the GPI keys have next_key_stride > B, a* covers 0 and A-1 and differs per policy."""
    gen = torch.Generator().manual_seed(1000 * variant + B + 7 * n_pol + 13 * K + seed)
    r = lambda *sh: torch.randn(*sh, generator=gen)
    c = dict(variant=variant, B=B, n_pol=n_pol, S=S, A=A, D=D, G=G if variant == 2 else 0, K=K if variant == 2 else 0,
             beta=2.5 if variant == 2 else 1.0, next_form=next_form)
    c['cur'] = r(n_pol, B, D)
    c['phis'] = torch.rand(B, D, generator=gen) * 2.5 - 1.5
    c['rs'] = r(B)
    c['gammas'] = torch.where(torch.rand(B, generator=gen) < 0.05, 0.0, 0.9)
    c['s'], c['s1'] = r(B, S), r(B, S)
    c['w_stride'] = D + 5
    c['w'] = r(n_pol, c['w_stride']) * 0.5
    gl = c['G'] * S + c['G'] + c['K'] * (2 * S + 1)
    c['g_stride'] = gl + 3
    c['g'] = (torch.rand(n_pol, c['g_stride'], generator=gen) * 2 - 1) / max(S, 1) ** 0.5
    if c['K']:
        c['g'][:, c['G'] * S + c['G']:gl] = r(n_pol, gl - c['G'] * S - c['G']) * 0.5
    c['h'] = (torch.rand(D * c['G'] + D, generator=gen) * 2 - 1) / max(c['G'], 1) ** 0.5
    if next_form == 'sel':
        c['nxt'] = r(n_pol, B, D)
    else:
        astar = torch.randint(0, A, (n_pol, B), generator=gen)
        astar[0::2, 0], astar[1::2, 0], astar[0::2, -1], astar[1::2, -1] = 0, A - 1, A - 1, 0
        c['key_stride'] = B + 5
        pad = torch.randint(0, A, (n_pol, 5), generator=gen)       # rows past B: valid actions the kernel must not read
        idx = torch.cat([astar, pad], 1)
        hi = torch.randint(0, 1 << 20, idx.shape, generator=gen)
        c['keys'] = (hi << 32) | (0xFFFFFFFF - idx)
        c['next_psi'] = r(B, n_pol, A * D)
        c['nxt'] = torch.stack([c['next_psi'][torch.arange(B), p].view(B, A, D)[torch.arange(B), astar[p]] for p in range(n_pol)])
    return c


def reference_of(c):
    """Per policy: (sum diff^2, sum e^2, dL/dcur, gradient row)."""
    S, D, G, K = c['S'], c['D'], c['G'], c['K']
    gl = G * S + G + K * (2 * S + 1)
    return [td_reference(c['variant'], c['cur'][p], c['nxt'][p], c['phis'], c['rs'], c['gammas'], c['w'][p, :D], c['A'], c['beta'],
                         c['g'][p, :gl], c['h'], c['s'], c['s1'], G, K) for p in range(c['n_pol'])]


def want_aux_of(c):
    S, D, G, K = c['S'], c['D'], c['G'], c['K']
    return 0 if c['variant'] == 0 else (D if c['variant'] == 1 else D + G * S + G + K * (2 * S + 1) + D * G + D)


def sfgpi_step_prep_mc(c, g_dev, h_dev):
    """M = Wh Wg and c = 2 (Wh bg + bh) of every policy from sfgpi_step_prep with only its TSF part enabled."""
    from deep_successor_features_for_transfer_b200.library import NetSpec
    S, A, D = c['S'], c['A'], c['D']
    pr = _lib.StepPrepArgs()
    pr.net = NetSpec([S, 256, 256, 256, A * D], ['none', 'relu', 'relu', 'none'], A, D).desc()
    mc = torch.full((c['n_pol'] * (D * S + D),), float('nan'), device='cuda')
    pr.tsf_g, pr.tsf_h, pr.tsf_mc = g_dev.data_ptr(), h_dev.data_ptr(), mc.data_ptr()
    pr.tsf_g_stride, pr.tsf_G, pr.tsf_lo, pr.tsf_n = c['g_stride'], c['G'], 0, c['n_pol']
    _lib.call('sfgpi_step_prep', C.byref(pr), stream())
    return mc


def run_td(c, mc=False, expect_rc=0):
    """
    One sfgpi_td_step call on device copies of c's inputs.  Before it, exactly the outputs the header says the launch writes are
    set to NaN -- d_out, loss_part, tsf_part and the first want_aux floats of the aux rows (all n_blocks rows in variant 1, slot 0
    in variant 2) -- and a sentinel tail sits behind every buffer (and in the aux floats / slots that are not written).  Returns
    the outputs as CPU tensors after checking that every written float is finite and every other one untouched.
    """
    v, B, n_pol, S, D = c['variant'], c['B'], c['n_pol'], c['S'], c['D']
    lib = _lib.lib()
    nblk = lib.sfgpi_td_partials(B)
    want_aux = want_aux_of(c)
    aux_len = want_aux + 3
    n_red = D + D * S + D + c['K'] * (2 * S + 1) if v == 2 else D
    dev = {k: c[k].cuda().contiguous() for k in ('cur', 'phis', 'rs', 'gammas', 's', 's1', 'w', 'g', 'h')}
    d_out_b, d_out = guarded(n_pol * B * D)
    loss_b, loss = guarded(n_pol * nblk * 2)
    aux_b, aux = guarded(n_pol * nblk * aux_len, SENTINEL)
    aux3 = aux.view(n_pol, nblk, aux_len)
    written = torch.zeros_like(aux3, dtype=torch.bool)
    if v == 1:
        written[:, :, :want_aux] = True
    elif v == 2:
        written[:, 0, :want_aux] = True
    aux3[written] = float('nan')
    tsf_b, tsf = guarded(n_pol * nblk * n_red) if v == 2 else (None, None)
    t = _lib.TdArgs()
    t.variant, t.n_pol, t.B, t.S, t.A, t.D, t.G, t.beta = v, n_pol, B, S, c['A'], D, c['G'], c['beta']
    t.cur_sel, t.phis, t.rs, t.gammas = (_lib.ptr(dev[k]) for k in ('cur', 'phis', 'rs', 'gammas'))
    t.states, t.next_states = _lib.ptr(dev['s']), _lib.ptr(dev['s1'])
    t.w, t.w_stride, t.g, t.g_stride, t.h, t.n_flows = _lib.ptr(dev['w']), c['w_stride'], _lib.ptr(dev['g']), c['g_stride'], _lib.ptr(dev['h']), c['K']
    if c['next_form'] == 'sel':
        dev['nxt'] = c['nxt'].cuda().contiguous()
        t.next_sel = _lib.ptr(dev['nxt'])
    else:
        dev['next_psi'], dev['keys'] = c['next_psi'].cuda().contiguous(), c['keys'].cuda().contiguous()
        t.next_psi, t.next_keys, t.next_key_stride = _lib.ptr(dev['next_psi']), _lib.ptr(dev['keys']), c['key_stride']
    t.d_out, t.loss_part, t.aux_grad_part, t.aux_len = _lib.ptr(d_out), _lib.ptr(loss), _lib.ptr(aux), aux_len
    t.tsf_part = _lib.ptr(tsf)
    if mc:
        dev['mc'] = sfgpi_step_prep_mc(c, dev['g'], dev['h'])
        t.tsf_mc = _lib.ptr(dev['mc'])
    rc = lib.sfgpi_td_step(C.byref(t), stream())
    torch.cuda.synchronize()
    assert rc == expect_rc, f'rc {rc}: {lib.sfgpi_last_error().decode()}'
    if rc != 0:                                                    # refused: nothing may have been launched
        for buf, n in ((d_out_b, d_out.numel()), (loss_b, loss.numel()), (tsf_b, 0 if tsf is None else tsf.numel())):
            if buf is not None:
                assert torch.isnan(buf[:n]).all() and (buf[n:] == SENTINEL).all()
        return lib.sfgpi_last_error().decode()
    for buf, n, name in ((d_out_b, d_out.numel(), 'd_out'), (loss_b, loss.numel(), 'loss_part'),
                         (tsf_b, 0 if tsf is None else tsf.numel(), 'tsf_part'), (aux_b, aux.numel(), 'aux_grad_part')):
        if buf is None:
            continue
        assert (buf[n:] == SENTINEL).all(), f'{name}: the launch wrote past the end of the buffer'
        if name != 'aux_grad_part':
            assert torch.isfinite(buf[:n]).all(), f'{name}: floats the launch must write are left unwritten (or not finite)'
    assert torch.isfinite(aux3[written]).all(), 'aux_grad_part: floats the launch must write are left unwritten (or not finite)'
    assert (aux3[~written] == SENTINEL).all(), 'aux_grad_part: the launch wrote outside its gradient rows'
    return dict(d_out=d_out.view(n_pol, B, D).cpu(), loss=loss.view(n_pol, nblk, 2).cpu(), aux=aux3.cpu(),
                tsf=None if tsf is None else tsf.cpu(), want_aux=want_aux)


def check_against_reference(c, out, what='', tol=TOL):
    v, D = c['variant'], c['D']
    ref = reference_of(c)
    assert err(out['d_out'], torch.stack([r[2] for r in ref])) < tol, f'{what} d_out'
    for p, (l1s, l2s, _, row) in enumerate(ref):
        lp = out['loss'][p].double().sum(0)
        assert abs(float(lp[0]) - l1s) <= tol * l1s, f'{what} policy {p}: sum diff^2 {float(lp[0])} vs {l1s}'
        if v == 0:
            assert float(lp[1]) == 0.0
            continue
        assert abs(float(lp[1]) - l2s) <= tol * l2s, f'{what} policy {p}: sum e^2 {float(lp[1])} vs {l2s}'
        got = out['aux'][p, :, :D].double().sum(0) if v == 1 else out['aux'][p, 0, :out['want_aux']]
        assert_row_close(got, row, row_blocks(v, D, c['S'], c['G'], c['K']), f'{what} policy {p}', tol)


def assert_same_bits(a, b):
    for k in ('d_out', 'loss', 'aux', 'tsf'):
        if a[k] is not None:
            assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), f'{k} differs'


BATCHES = [1, 31, 32, 33, 255, 256, 257, 1000, 2049]


@pytest.mark.gpu
@pytest.mark.parametrize('n_pol', [1, 3])
@pytest.mark.parametrize('B', BATCHES)
@pytest.mark.parametrize('next_form', ['sel', 'psi'])
@pytest.mark.parametrize('variant', [0, 1, 2])
def test_td_step_vs_float64(variant, next_form, B, n_pol):
    """Every variant and next-value form at the batch edges: 1 row before 7 empty CTAs, a CTA edge, a cluster edge, a last
    cluster of one row (257, 2049); two launches give the same bits."""
    c = make_td_case(variant, B, n_pol, next_form=next_form)
    out = run_td(c)
    check_against_reference(c, out)
    assert_same_bits(out, run_td(c))


TSF_SHAPES = [(4, 12, 100, 0), (11, 50, 100, 0), (4, 12, 100, 3), (4, 12, 16, 10), (1, 1, 1, 0)]


@pytest.mark.gpu
@pytest.mark.parametrize('B', [33, 257])
@pytest.mark.parametrize('next_form', ['sel', 'psi'])
@pytest.mark.parametrize('S,D,G,K', TSF_SHAPES)
def test_td_step_tsf_shapes(S, D, G, K, next_form, B):
    """Variant 2 at every TSF shape, M and c derived in every CTA (tsf_mc NULL) and taken from sfgpi_step_prep: the two give the
    same bits (the prologue runs the same dot products in the same order)."""
    A = 27 if D == 50 else 9
    c = make_td_case(2, B, 3, S=S, A=A, D=D, G=G, K=K, next_form=next_form)
    own = run_td(c)
    check_against_reference(c, own, 'tsf_mc NULL:')
    assert_same_bits(own, run_td(c, mc=True))


def _largest(fn, lo, hi, limit):
    """Largest x in [lo, hi) with fn(x) <= limit (fn increasing)."""
    return max(x for x in range(lo, hi) if fn(x) <= limit)


def td_edge_sizes(variant):
    """(parameter, bytes) at the shared-memory edges: largest <= 48 KB, smallest above, largest accepted, first refused.
    Variant 1 steps D (520 B a step); variant 2 steps G at S = D = 1 with M and c derived in the kernel (12 B a step)."""
    fn = (lambda D: td_smem_bytes(1, D)) if variant == 1 else (lambda G: td_smem_bytes(2, 1, 1, G))
    top = KMAX_SMEM - TD_STATIC_SMEM
    x48 = _largest(fn, 1, 100000, 48 * 1024)
    xmax = _largest(fn, 1, 100000, top)
    return [(x48, fn(x48)), (x48 + 1, fn(x48 + 1)), (xmax, fn(xmax))], (xmax + 1, fn(xmax + 1))


def td_edge_case(variant, x):
    return make_td_case(1, 257, 1, D=x) if variant == 1 else make_td_case(2, 257, 1, S=1, A=3, D=1, G=x)


@pytest.mark.gpu
@pytest.mark.parametrize('edge', [0, 1, 2])
@pytest.mark.parametrize('variant', [1, 2])
def test_td_step_smem_edges(variant, edge):
    """Launches right below and above the 48 KB default and at the largest size the host accepts (static shared memory
    included) run and match float64."""
    x, nbytes = td_edge_sizes(variant)[0][edge]
    assert (nbytes <= 48 * 1024) == (edge == 0) and nbytes + TD_STATIC_SMEM <= KMAX_SMEM
    c = td_edge_case(variant, x)
    # variant 2 reaches these sizes through G in the thousands: M and c are fp32 dot products of that length, whose rounding
    # grows like sqrt(G) ulps
    check_against_reference(c, run_td(c), f'{nbytes} B:', TOL if variant == 1 else 1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize('variant', [1, 2])
def test_td_step_smem_refused(variant):
    x, nbytes = td_edge_sizes(variant)[1]
    assert nbytes + TD_STATIC_SMEM > KMAX_SMEM
    msg = run_td(td_edge_case(variant, x), expect_rc=E_SMEM)
    assert str(nbytes) in msg


# ---- sfgpi_target_adapt at its shared-memory edges ------------------------------------------------------------------------------
def adapt_smem_bytes(N, G, D):
    return 4 * (2 * N + N * G + 2 * G + 4 * D)                     # csrc/target.cu, sfgpi_target_adapt


def adapt_reference(c):
    """update_test_reward_mapper's loss (OracleSF.target_adapt_step) in float64 on given psi / next_psi: (loss, l2, l1, gw, gomega)."""
    f = lambda x: x.double()
    N, A, D, G, S = c['N'], c['A'], c['D'], c['G'], c['S']
    w, om = f(c['w']).requires_grad_(True), f(c['om']).requires_grad_(True)
    norm = om / om.sum()
    g = f(c['g'])
    Wg, bg = g[:, :G * S].view(N, G, S), g[:, G * S:G * S + G]
    ts, ts1 = torch.einsum('ngs,s->ng', Wg, f(c['s'])) + bg, torch.einsum('ngs,s->ng', Wg, f(c['s1'])) + bg
    Wh, bh = f(c['h'])[:D * G].view(D, G), f(c['h'])[D * G:]
    aff = Wh @ (norm[:, None] * ts).sum(0) + bh + Wh @ (norm[:, None] * ts1).sum(0) + bh
    tphi = f(c['phi']) * aff
    tsf = (norm[:, None] * f(c['psi'])[:, c['a']]).sum(0)
    ntsf = (norm[:, None] * f(c['next_psi'])[:, c['a1']]).sum(0)
    l1 = ((tsf - (tphi + c['gamma'] * ntsf)) ** 2).mean()
    l2 = ((w * tphi).sum() - c['r']) ** 2
    loss = l1 + c['beta'] * l2 + c['l1_coef'] * om.abs().sum()
    gw, go = torch.autograd.grad(loss, [w, om])
    return float(loss.detach()), float(l2.detach()), float(l1.detach()), gw, go


def run_adapt(N, G, D=12, S=4, A=5, expect_rc=0):
    gen = torch.Generator().manual_seed(N * 7919 + G)
    r = lambda *sh: torch.randn(*sh, generator=gen)
    c = dict(N=N, A=A, D=D, G=G, S=S, psi=r(N, A, D), next_psi=r(N, A, D), g=(torch.rand(N, G * S + G, generator=gen) * 2 - 1) * 0.5,
             h=(torch.rand(D * G + D, generator=gen) * 2 - 1) / G ** 0.5, s=r(S), s1=r(S), phi=r(D), r=0.7, gamma=0.9, a=1, a1=A - 1,
             beta=2.0, l1_coef=0.01, w=r(D) * 0.5, om=torch.rand(N, generator=gen) + 0.5)
    d = {k: c[k].cuda().contiguous() for k in ('psi', 'next_psi', 'g', 'h', 's', 's1', 'phi', 'w', 'om')}
    z = lambda n, dt=torch.float32: torch.zeros(n, dtype=dt, device='cuda')
    d.update(w_m=z(D), w_v=z(D), o_m=z(N), o_v=z(N), step=z(1, torch.int32), epoch=z(1, torch.int32))
    losses_b, losses = guarded(3)
    a = _lib.TargetArgs()
    a.N, a.A, a.D, a.G, a.S = N, A, D, G, S
    a.psi, a.next_psi, a.g, a.g_stride, a.h = _lib.ptr(d['psi']), _lib.ptr(d['next_psi']), _lib.ptr(d['g']), G * S + G, _lib.ptr(d['h'])
    a.s, a.s1, a.phi, a.r, a.gamma, a.a, a.a1 = _lib.ptr(d['s']), _lib.ptr(d['s1']), _lib.ptr(d['phi']), c['r'], c['gamma'], c['a'], c['a1']
    a.beta, a.l1_coef, a.lr_w, a.wd_w, a.lr_omega, a.wd_omega, a.lr_omega_decay = c['beta'], c['l1_coef'], 1e-3, 0.0, 1e-3, 0.0, 0.0
    a.w, a.omegas, a.w_m, a.w_v, a.o_m, a.o_v = (_lib.ptr(d[k]) for k in ('w', 'om', 'w_m', 'w_v', 'o_m', 'o_v'))
    a.step, a.epoch, a.losses = _lib.ptr(d['step']), _lib.ptr(d['epoch']), _lib.ptr(losses)
    lib = _lib.lib()
    rc = lib.sfgpi_target_adapt(C.byref(a), stream())
    torch.cuda.synchronize()
    assert rc == expect_rc, f'rc {rc}: {lib.sfgpi_last_error().decode()}'
    if rc != 0:
        assert torch.isnan(losses).all() and int(d['step'][0]) == 0 and torch.equal(d['w'].cpu(), c['w'])
        return lib.sfgpi_last_error().decode()
    assert (losses_b[3:] == SENTINEL).all() and int(d['step'][0]) == 1 and int(d['epoch'][0]) == 1
    loss, l2, l1, gw, go = adapt_reference(c)
    for got, ref in zip(losses.cpu().tolist(), (loss, l2, l1)):
        assert abs(got - ref) <= TOL * abs(ref)
    # first Adam step (m = 0.1 g, v = 0.001 g^2, bias corrections 0.1 and 0.001): p - lr g / (|g| + eps); omegas clamped >= 1e-7
    w_want = c['w'].double() - 1e-3 * gw / (gw.abs() + 1e-8)
    om_want = (c['om'].double() - 1e-3 * go / (go.abs() + 1e-8)).clamp_min(1e-7)
    assert (d['w'].cpu().double() - w_want).abs().max() < 1e-6
    assert (d['om'].cpu().double() - om_want).abs().max() < 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize('edge', [0, 1, 2, 3])
def test_target_adapt_smem_edges(edge):
    """sfgpi_target_adapt (N * G floats of shared memory) right below and above 48 KB, at the largest size the host accepts, and
    one step beyond, which is refused with SFGPI_E_SMEM before anything is launched."""
    N, D = 2, 12
    fn = lambda G: adapt_smem_bytes(N, G, D)
    g48 = _largest(fn, 1, 100000, 48 * 1024)
    gmax = _largest(fn, 1, 100000, KMAX_SMEM - ADAPT_STATIC_SMEM)
    G = [g48, g48 + 1, gmax, gmax + 1][edge]
    if edge < 3:
        run_adapt(N, G, D)
    else:
        assert str(fn(G)) in run_adapt(N, G, D, expect_rc=E_SMEM)


# ---- the TD step inside the real train step -------------------------------------------------------------------------------------
PRECISIONS = ['fp32', 'bf16', 'tf32', 'tf32x3']
N_LIB = 3


def build_library(case, env, precision):
    from deep_successor_features_for_transfer_b200 import tsfdqn_nf
    from deep_successor_features_for_transfer_b200.workloads import ENVS, HYPER, ShapeTask, build_sf_library, build_tsf_agent, model_lambda
    if case in ('g1', 'g2'):
        return build_sf_library(env, N_LIB, precision=precision, seed=21)._library
    if case == 'g3':
        return build_tsf_agent(env, N_LIB, beta=2.5, precision=precision, seed=21)[0]._library
    shp = ENVS[env]
    torch.manual_seed(21)
    hp = dict(HYPER, g_h_function_dims=100, beta_loss_coefficient=2.5, n_coupling_layers=3, precision=precision)
    sf = tsfdqn_nf.DeepTSF(model_lambda([256, 256], ['relu', 'relu']), hyperparameters=hp)
    ag = tsfdqn_nf.TSFDQN(deep_sf=sf, buffer_handle=lambda: tsfdqn_nf.ReplayBuffer(), gamma=0.9, T=500, encoding=None, hyperparameters=hp)
    ag.reset()
    for i in range(N_LIB):
        ag.add_training_task(ShapeTask(shp['S'], shp['A'], shp['D'], i))
    return sf._library


@pytest.mark.gpu
@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('env,B', [('reacher', 257), ('hopper', 257)])
@pytest.mark.parametrize('policy', [1, 'all'])
@pytest.mark.parametrize('case', ['g1', 'g2', 'g3', 'nf'])
def test_train_step_td_vs_float64(case, policy, env, B, precision):
    """
    The TD step as the train step runs it (tensor-core modes: next values gathered from next_psi by the GPI keys; bf16: M and c
    from the prologue, expand as rider CTAs of the dgrad launch) against float64 on the step's own gathered inputs, and a
    relaunch of the step's TD arguments on the pre-step w, g, h with the expand as its own launch gives the same bits.
    """
    lib = build_library(case, env, precision)
    sp = lib.spec
    S, A, D = sp.dims[0], sp.n_actions, sp.n_features
    variant = {'g1': 0, 'g2': 1, 'g3': 2, 'nf': 2}[case]
    gen = torch.Generator().manual_seed(5 + B)
    tr = [x.cuda() for x in synthetic_transitions(B, S, A, D, gen, hopper=env == 'hopper')]
    states, actions, rs, phis, next_states, gammas = tr
    w0 = lib.w.clone()
    g0, h0 = (lib.g.clone(), lib.h.clone()) if variant == 2 else (None, None)
    beta = 2.5 if variant == 2 else 1.0                          # (variants 0 and 1 have no loss coefficient)
    if variant == 0:
        lib.train_step((states, actions, phis, next_states, gammas), policy, True, variant=0)
    else:
        lib.train_step(tuple(tr), policy, True, variant=variant, beta=beta)
    torch.cuda.synchronize()
    plan = lib._ws[lib.last_plan_key]
    ws, t, n_pol, lo = plan['ws'], plan['t'], plan['n_pol'], plan['lo']
    assert bool(t.next_psi) == (precision != 'fp32')
    if precision == 'fp32':
        nxt = ws['next_sel']
    else:
        keys = plan['keys'][:n_pol]
        astar = (0xFFFFFFFF - (keys & 0xFFFFFFFF)).cpu()
        npsi = ws['next_psi'].cpu().view(B, n_pol, A, D)
        nxt = torch.stack([npsi[torch.arange(B), p, astar[p]] for p in range(n_pol)])
    K = lib.n_flows if variant == 2 else 0
    G = lib.G if variant == 2 else 0
    gl = lib.g.shape[1] if variant == 2 else 0
    want_aux = ws['aux_len']
    out = dict(d_out=ws['d_out'].cpu(), loss=ws['loss_part'].cpu(), want_aux=want_aux,
               aux=ws['aux_part'].cpu(), tsf=ws['tsf_part'].cpu() if variant == 2 else None)
    for p in range(n_pol):
        l1s, l2s, dcur, row = td_reference(variant, ws['cur_sel'][p], nxt[p], phis, rs, gammas, w0[lo + p], A, beta,
                                           g0[lo + p] if variant == 2 else None, h0, states, next_states, G, K)
        assert err(out['d_out'][p], dcur) < TOL
        lp = out['loss'][p].double().sum(0)
        assert abs(float(lp[0]) - l1s) <= TOL * l1s
        if variant:
            assert abs(float(lp[1]) - l2s) <= TOL * l2s
            got = out['aux'][p, :, :D].double().sum(0) if variant == 1 else out['aux'][p, 0, :want_aux]
            assert_row_close(got, row, row_blocks(variant, D, S, G, K), f'policy {lo + p}')
    # relaunch: pre-step w, g, h, fresh outputs, the expand as its own launch
    t2 = _lib.TdArgs.from_buffer_copy(t)
    t2.defer_expand = 0
    t2.w = w0[lo].data_ptr()
    if variant == 2:
        t2.g, t2.h = g0[lo].data_ptr(), h0.data_ptr()
    fresh = {k: torch.full_like(ws[k], float('nan')) for k in ('d_out', 'loss_part', 'aux_part') + (('tsf_part',) if variant == 2 else ())}
    t2.d_out, t2.loss_part, t2.aux_grad_part = (fresh[k].data_ptr() for k in ('d_out', 'loss_part', 'aux_part'))
    if variant == 2:
        t2.tsf_part = fresh['tsf_part'].data_ptr()
    _lib.call('sfgpi_td_step', C.byref(t2), stream())
    torch.cuda.synchronize()
    again = dict(d_out=fresh['d_out'].cpu(), loss=fresh['loss_part'].cpu(), aux=fresh['aux_part'].cpu(),
                 tsf=fresh['tsf_part'].cpu() if variant == 2 else None)
    if variant == 2:                                               # only slot 0 of the aux rows is written in variant 2
        out['aux'], again['aux'] = out['aux'][:, 0, :want_aux].contiguous(), again['aux'][:, 0, :want_aux].contiguous()
    elif variant == 0:
        out['aux'] = again['aux'] = None
    assert_same_bits(out, again)


# ---- the other two loss heads that feed Adam partials ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('B', [1, 255, 256, 257, 1000])
def test_phi_head_vs_float64(B):
    """sfgpi_phi_head: e = w.phi - r, d_out = (2/B) e w, per-CTA partials of dL/dw and of sum e^2 (one CTA per 256 rows)."""
    D = 13
    gen = torch.Generator().manual_seed(B)
    phi, w, r = torch.randn(B, D, generator=gen), torch.randn(D, generator=gen) * 0.5, torch.randn(B, generator=gen)
    lib = _lib.lib()
    nblk = lib.sfgpi_phi_head_partials(B)
    d_b, d_out = guarded(B * D)
    dw_b, dw = guarded(nblk * D)
    l_b, lp = guarded(nblk * 2)
    pd, wd, rd = phi.cuda(), w.cuda(), r.cuda()
    rc = lib.sfgpi_phi_head(_lib.ptr(pd), _lib.ptr(wd), _lib.ptr(rd), B, D, _lib.ptr(d_out), _lib.ptr(dw), _lib.ptr(lp), stream())
    torch.cuda.synchronize()
    assert rc == 0, lib.sfgpi_last_error().decode()
    for buf, n in ((d_b, B * D), (dw_b, nblk * D), (l_b, nblk * 2)):
        assert torch.isfinite(buf[:n]).all() and (buf[n:] == SENTINEL).all()
    ph, wl = phi.double().requires_grad_(True), w.double().requires_grad_(True)
    e = ph @ wl - r.double()
    loss = (e ** 2).mean()
    gphi, gw = torch.autograd.grad(loss, [ph, wl])
    assert err(d_out.view(B, D).cpu(), gphi) < TOL
    assert err(dw.view(nblk, D).cpu().double().sum(0), gw) < TOL
    lpc = lp.view(nblk, 2).cpu().double()
    assert (lpc[:, 0] == 0).all()
    assert abs(float(lpc[:, 1].sum()) - float((e ** 2).sum())) <= TOL * float((e ** 2).sum())


def g4_args(B, A, D, seed=0):
    gen = torch.Generator().manual_seed(B + seed)
    r = lambda *sh: torch.randn(*sh, generator=gen)
    c = dict(cur=r(B, D), nxt=r(B, D), phi=r(B, D), rs=r(B), gammas=torch.full((B,), 0.9), w=r(D) * 0.5, bias=r(1), coef=torch.tensor([0.7]))
    d = {k: v.cuda() for k, v in c.items()}
    outs = dict(d_psi=guarded(B * D), d_phi=guarded(B * D), grad_small=guarded(D + 2), losses=guarded(4))
    a = _lib.G4Args()
    a.B, a.A, a.D = B, A, D
    a.cur_sel, a.next_sel, a.phi, a.rs, a.gammas, a.w, a.bias, a.coef = (_lib.ptr(d[k]) for k in ('cur', 'nxt', 'phi', 'rs', 'gammas', 'w', 'bias', 'coef'))
    a.d_psi, a.d_phi, a.grad_small, a.losses = (_lib.ptr(outs[k][1]) for k in ('d_psi', 'd_phi', 'grad_small', 'losses'))
    return a, c, outs, d


@pytest.mark.gpu
@pytest.mark.parametrize('B', [1, 32, 4096])
def test_g4_head_vs_float64(B):
    """sfgpi_g4_head: joint psi / phi loss with the learnable coefficient, every output against float64 autograd."""
    A, D = 5, 9
    a, c, outs, _ = g4_args(B, A, D)
    lib = _lib.lib()
    rc = lib.sfgpi_g4_head(C.byref(a), stream())
    torch.cuda.synchronize()
    assert rc == 0, lib.sfgpi_last_error().decode()
    for buf, view in outs.values():
        assert torch.isfinite(view).all() and (buf[view.numel():] == SENTINEL).all()
    f = lambda k: c[k].double()
    cur, phi, w, b, coef = (f(k).requires_grad_(True) for k in ('cur', 'phi', 'w', 'bias', 'coef'))
    psi_loss = ((cur - (phi + f('gammas')[:, None] * f('nxt'))) ** 2).sum() / (B * A * D)
    phi_loss = ((phi @ w + b - f('rs')) ** 2).mean()
    loss = phi_loss + coef[0] * psi_loss
    gcur, gphi, gw, gb, gc = torch.autograd.grad(loss, [cur, phi, w, b, coef])
    assert err(outs['d_psi'][1].view(B, D).cpu(), gcur) < TOL
    assert err(outs['d_phi'][1].view(B, D).cpu(), gphi) < TOL
    gs = outs['grad_small'][1].cpu().double()
    assert err(gs[:D], gw) < TOL
    assert abs(float(gs[D]) - float(gb)) <= TOL * max(abs(float(gb)), float(gw.abs().max()))
    assert abs(float(gs[D + 1]) + float(gc)) <= TOL * abs(float(gc))          # Adam maximises the coefficient: -dL/dc
    want = [float(loss), float(psi_loss), float(phi_loss), 0.7]
    for got, ref in zip(outs['losses'][1].cpu().tolist(), want):
        assert abs(got - ref) <= TOL * abs(ref)


@pytest.mark.gpu
def test_g4_head_refuses_b4097():
    a, _, outs, _ = g4_args(4097, 5, 9)
    assert _lib.lib().sfgpi_g4_head(C.byref(a), stream()) == E_INVALID
    torch.cuda.synchronize()
    assert torch.isnan(outs['d_psi'][1]).all() and torch.isnan(outs['losses'][1]).all()
