"""
-m gpu: the tensor-core (tcgen05, bf16 operands / fp32 accumulate) mode against the fp32 CPU oracle.
Stated tolerance (include/sfgpi.h, SURVEY section 7 "fp32 1e-5 parity vs tensor cores"): BF16_TOL = 2e-2 scale-relative
on psi / q, relative Frobenius error < 1e-2; GPI argmax must agree wherever the fp32 top-1/top-2 gap exceeds
BF16_TOL * max|q| (ties inside tolerance may flip).
"""
import numpy as np
import pytest
import torch

from oracle.sf_oracle import OracleSF, synthetic_transitions
from tests.golden_util import rel_err
from tests import gpu_util as gu

pytestmark = pytest.mark.gpu
BF16_TOL = 2e-2
HYPER_BF16 = dict(gu.HYPER, precision='bf16')


def fro_err(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def make(S, A, D, N, seed, tsf_dim=None, beta=1):
    gen = torch.Generator().manual_seed(seed)
    o = OracleSF(S, A, D, (256, 256), ('relu', 'relu'), tsf_dim=tsf_dim, beta=beta)
    for _ in range(N):
        o.add_random_policy(gen)
    return o, gen


@pytest.mark.parametrize('S,A,D,N,B,hopper', [
    (4, 9, 12, 4, 4096, False),          # 128 tiles: one tile per CTA (no ping-pong partner)
    (4, 9, 12, 6, 33 * 128 - 5, False),  # 198 tiles: paired mode, odd tile count per policy, ragged last tile
    (4, 9, 12, 10, 33 * 128 - 5, False), # 330 tiles: ping-pong pairs and single tiles, 33 tiles per policy
    (11, 27, 50, 5, 8192, True),         # Hopper on ping-pong pairs: output layer in 6 chunks, 64 tiles per policy
    (11, 27, 50, 3, 1000, True),         # Hopper: output layer in 6 chunks of <= 256 columns, S = 11
    (4, 2, 20, 3, 32, False),            # CartPole, a single partial tile
])
def test_bf16_forward_gpi_vs_oracle(S, A, D, N, B, hopper):
    _bf16_forward_gpi_vs_oracle(S, A, D, N, B, hopper)


@pytest.mark.parametrize('S,A,D,N,B,hopper', [
    (4, 9, 12, 6, 33 * 128 - 5, False),  # 198 tiles on 148 CTAs: two tiles on some CTAs (prefetch + early staging of the next tile)
    (4, 9, 12, 10, 33 * 128 - 5, False), # 330 tiles: up to three tiles per CTA
    (11, 27, 50, 5, 2048, True),         # Hopper: 6 output chunks alternate the two accumulators, S = 11 (two staged k-chunks)
])
def test_bf16_forward_chain_kernel_multi_tile(S, A, D, N, B, hopper):
    """The layer-pipelined single-tile kernel (csrc/mlp_chain_tc.cu) forced onto launches of more than one wave -- by default it
    only takes launches of <= 148 tiles, which the cases of test_bf16_forward_gpi_vs_oracle with few tiles already cover."""
    from deep_successor_features_for_transfer_b200 import _lib
    old = _lib.lib().sfgpi_set_option(b'forward_chain', 2)
    try:
        _bf16_forward_gpi_vs_oracle(S, A, D, N, B, hopper)
    finally:
        _lib.lib().sfgpi_set_option(b'forward_chain', old)


@pytest.mark.parametrize('variant', ['g2', 'g3'])
def test_bf16_chain_and_pair_kernels_agree_bit_for_bit(variant):
    """Both forward kernels issue the same MMAs in the same k order on the same bf16 operands and share the epilogue arithmetic:
    an all-task train step (online forward with saved activations / ReLU masks, fused GPI with 4 reward vectors, target
    forward) must leave bit-identical losses, weights and Adam moments whichever kernel ran the forward."""
    from deep_successor_features_for_transfer_b200 import _lib
    S, A, D, N, B = 4, 9, 12, 4, 1000
    tsf = variant == 'g3'
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N, gdim=100, beta=1, use_gpi=True)
    outs = []
    for mode in (0, 2):
        old = _lib.lib().sfgpi_set_option(b'forward_chain', mode)
        try:
            o, gen = make(S, A, D, N, seed=5, tsf_dim=100 if tsf else None)
            if tsf:
                sf, ag = gu.build_g3(meta, oracle=o)
                sf._library.set_precision('bf16')
            else:
                sf = ag = gu.build_g2(meta, oracle=o, hyper=HYPER_BF16)
            losses = [ag.update_successor_all(gu.cuda_tr(synthetic_transitions(B, S, A, D, gen)), use_gpi=True).clone() for _ in range(3)]
            lib = sf._library
            outs.append((torch.stack(losses).cpu(), lib.online[:N].clone().cpu(), lib.m[:N].clone().cpu(), lib.w[:N].clone().cpu()))
        finally:
            _lib.lib().sfgpi_set_option(b'forward_chain', old)
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def _bf16_forward_gpi_vs_oracle(S, A, D, N, B, hopper):
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make(S, A, D, N, seed=21)
    sf = gu.build_g2(meta, oracle=o, hyper=HYPER_BF16)
    assert sf._library.precision == 'bf16'
    x = synthetic_transitions(B, S, A, D, gen, hopper=hopper)[0]
    psi_ref = o.get_successors(x)
    psi = sf.get_successors(x.cuda()).cpu()
    assert rel_err(psi, psi_ref) < BF16_TOL and fro_err(psi, psi_ref) < 1e-2
    psi_t = sf._library.forward_psi(x.cuda(), 1, 1, target=True).cpu()
    assert fro_err(psi_t[:, 0], psi_ref[:, 1]) < 1e-2
    q_ref, task_ref = o.GPI(x, 1)
    q, task = sf.GPI(x.cuda(), 1)
    assert rel_err(q.cpu(), q_ref) < BF16_TOL
    ok, nbad = gu.argmax_mismatch_ok(q_ref, task_ref, task.cpu(), 'task', BF16_TOL)
    assert ok, f'{nbad} task mismatches outside tolerance'
    _, key_a, key_t = sf._library.gpi(x.cuda(), sf.fit_w[1].weight, want_q=False)
    act, val = sf._library.decode_keys(key_a, want_value=True)
    act_ref = torch.argmax(torch.max(q_ref, dim=1).values, dim=-1)
    ok, nbad = gu.argmax_mismatch_ok(q_ref, act_ref, act.cpu(), 'action', BF16_TOL)
    assert ok, f'{nbad} action mismatches outside tolerance'
    # self-consistency (exact): keys agree with the q the same kernel returned
    assert torch.equal(val, q.reshape(B, -1).max(dim=1).values)
    assert torch.equal(act, torch.argmax(q.max(dim=1).values, dim=-1))
    assert torch.equal(sf._library.decode_keys(key_t), torch.argmax(q.max(dim=2).values, dim=1))


@pytest.mark.parametrize('variant,N', [('g2', 4), ('g3', 6)])
def test_bf16_train_step_vs_oracle(variant, N):
    S, A, D, B = 4, 9, 12, 4096
    tsf = variant == 'g3'
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N, gdim=100, beta=1, use_gpi=True)
    o, gen = make(S, A, D, N, seed=31, tsf_dim=100 if tsf else None)
    if tsf:
        sf, ag = gu.build_g3(meta, oracle=o)
        sf._library.set_precision('bf16')
    else:
        sf = ag = gu.build_g2(meta, oracle=o, hyper=HYPER_BF16)
    W_before = [W.clone() for W, _ in gu.psi_params(sf, 1)]
    tr = synthetic_transitions(B, S, A, D, gen)
    ref = o.tsf_update_successor(tr, 1, True) if tsf else o.update_successor(tr, 1, True)
    out = ag.update_successor(gu.cuda_tr(tr), 1, True)
    assert np.allclose([float(v) for v in out], [float(v) for v in ref], rtol=3e-2, atol=1e-6)
    for l, (W, _) in enumerate(gu.psi_params(sf, 1)):
        d_mine, d_ref = (W - W_before[l]).flatten().double(), (o.psi[1][l][0] - W_before[l]).flatten().double()
        cos = float(d_mine @ d_ref / (d_mine.norm() * d_ref.norm()))
        assert cos > 0.9, f'layer {l}: update direction cos {cos}'
    # all-task step with GPI over all reward vectors (n_w = N: the multi-vector epilogue)
    tr = synthetic_transitions(B, S, A, D, gen)
    ref = o.ensemble_update_frozen(tr, tsf=tsf, use_gpi=True)
    losses = ag.update_successor_all(gu.cuda_tr(tr), use_gpi=True).cpu()
    for i in range(N):
        assert np.allclose(losses[i].numpy(), [float(v) for v in ref[i]], rtol=3e-2, atol=1e-6)


def _rb(t):
    """Straight-through bf16 rounding: the value the tensor core consumes, the fp32 gradient path."""
    return t + (t.bfloat16().float() - t).detach()


def torch_psi_grads(o, lo, n_pol, x, actions, d_out, emulate_bf16=False):
    """
    Autograd reference of PackedSFLibrary.psi_gradients: list over policies of [(dW_l, db_l)].  emulate_bf16 rounds the
    operands of every GEMM (inputs, weights, stored activations) to bf16 exactly where the tensor-core forward does, so the
    ReLU masks are the ones the kernels see: a mask that flips because a pre-activation sits within bf16 noise of zero is
    a full-size element error (relative Frobenius error = sqrt(fraction flipped), ~5 % at 0.3 % flips) and says nothing
    about the backward kernels.
    """
    from oracle.sf_oracle import act_fn
    out = []
    B = x.shape[0]
    rb = _rb if emulate_bf16 else (lambda t: t)
    for p in range(n_pol):
        layers = [(W.clone().requires_grad_(True), b.clone().requires_grad_(True)) for W, b in o.psi[lo + p]]
        h = rb(x)
        for (W, b), a in zip(layers, o.acts):
            h = act_fn(a)(torch.addmm(b, h, rb(W).t()))
            if W is not layers[-1][0]:
                h = rb(h)
        psi = h.view(B, o.A, o.D)
        (psi[torch.arange(B), actions] * d_out[p]).sum().backward()
        out.append([(W.grad, b.grad) for W, b in layers])
    return out


@pytest.mark.parametrize('precision,tol', [('bf16', 1.5e-2), ('fp32', 2e-5)])
@pytest.mark.parametrize('S,A,D,N,B,hopper', [
    (4, 9, 12, 3, 1000, False),          # Reacher: one output-layer chunk (K = 112), ragged last tile, 2 batch splits
    (4, 9, 12, 5, 33 * 128 - 5, False),  # paired tiles in the dgrad kernel
    (11, 27, 50, 2, 300, True),          # Hopper: 6 output-layer chunks in dgrad, 11 output tiles in wgrad, S = 11
    (4, 2, 20, 2, 32, False),            # CartPole shape, half a tile
])
def test_psi_backward_vs_autograd(precision, tol, S, A, D, N, B, hopper):
    """The backward kernels alone (tensor-core and fp32) against torch autograd on the oracle's weights."""
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make(S, A, D, N, seed=77)
    sf = gu.build_g2(meta, oracle=o, hyper=dict(gu.HYPER, precision=precision))
    lib = sf._library
    tr = synthetic_transitions(B, S, A, D, gen, hopper=hopper)
    x, actions = tr[0], tr[1]
    lo, n_pol = (1, N - 1)
    d_out = torch.randn(n_pol, B, D, generator=gen) * 1e-4
    ref = torch_psi_grads(o, lo, n_pol, x, actions, d_out, emulate_bf16=precision == 'bf16')
    got = lib.psi_gradients(x.cuda(), actions.cuda(), d_out.cuda(), lo, n_pol).cpu()
    for p in range(n_pol):
        for l, ((W, b), (gW, gb)) in enumerate(zip(lib.spec.views(got[p]), ref[p])):
            assert fro_err(W, gW) < tol, f'policy {p} layer {l}: dW error {fro_err(W, gW)}'
            assert fro_err(b, gb) < tol, f'policy {p} layer {l}: db error {fro_err(b, gb)}'


def test_bf16_forward_unit_table_schedule():
    """380 row tiles on 148 SMs: the balanced pairs + singles schedule (unit table) of the one-CTA-per-SM kernel."""
    _bf16_forward_gpi_vs_oracle(4, 9, 12, 10, 38 * 128 - 5, False)


@pytest.mark.parametrize('S,A,D,N,B', [(4, 9, 12, 3, 1000), (11, 27, 50, 2, 333)])
def test_step_prep_equals_separate_passes(S, A, D, N, B):
    """sfgpi_step_prep (one launch) == sfgpi_pack_bf16 x2 + sfgpi_keys_fill + sfgpi_fold_gpi + build_xo, bit for bit."""
    import ctypes as C
    from deep_successor_features_for_transfer_b200 import _lib
    from deep_successor_features_for_transfer_b200.library import _stream
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make(S, A, D, N, seed=31)
    sf = gu.build_g2(meta, oracle=o, hyper=HYPER_BF16)
    lib = sf._library
    lib.target[:N].mul_(1.5)                                    # online != target
    desc = lib.spec.desc()
    x = synthetic_transitions(B, S, A, D, gen)[0].cuda()
    nq = _lib.lib().sfgpi_gpi_fold_rows(C.byref(desc), N)
    st = _stream()
    # separate passes
    lib._pack('online', 0, N)
    lib._pack('target', 1, N - 1)
    ref_on, ref_tg = lib._shadow_for('online').clone(), lib._shadow_for('target').clone()
    keys_ref = torch.zeros(5, B, dtype=torch.int64, device='cuda')
    _lib.call('sfgpi_keys_fill', keys_ref.data_ptr(), keys_ref.numel() - 1, st)
    wq_ref = torch.zeros(N * nq * 256, dtype=torch.bfloat16, device='cuda')
    bq_ref = torch.zeros(N * nq, device='cuda')
    _lib.call('sfgpi_fold_gpi', C.byref(desc), lib.online.data_ptr(), 0, N, lib.w.data_ptr(), N, 0, wq_ref.data_ptr(),
              bq_ref.data_ptr(), st)
    xo_ref = torch.zeros(B, 64, device='cuda')
    xo_ref[:, :S] = x
    xo_ref[:, S] = 1.0
    xo_ref = xo_ref.to(torch.bfloat16)
    # one launch
    lib._shadow_for('online').zero_()
    lib._shadow_for('target').zero_()
    keys = torch.zeros(5, B, dtype=torch.int64, device='cuda')
    wq, bq = torch.zeros_like(wq_ref), torch.zeros_like(bq_ref)
    xo = torch.zeros(B, 64, dtype=torch.bfloat16, device='cuda')
    pr = _lib.StepPrepArgs()
    pr.net = desc
    pr.pack_params[0], pr.pack_out[0], pr.pack_lo[0], pr.pack_n[0] = lib.online.data_ptr(), lib._shadow_for('online').data_ptr(), 0, N
    pr.pack_params[1], pr.pack_out[1], pr.pack_lo[1], pr.pack_n[1] = lib.target.data_ptr(), lib._shadow_for('target').data_ptr(), 1, N - 1
    pr.keys, pr.n_keys = keys.data_ptr(), keys.numel() - 1
    pr.fold_params, pr.fold_lo, pr.fold_n = lib.online.data_ptr(), 0, N
    pr.w, pr.n_w, pr.w_diag, pr.wq, pr.bq = lib.w.data_ptr(), N, 0, wq.data_ptr(), bq.data_ptr()
    pr.x, pr.B, pr.xo_bf16 = x.data_ptr(), B, xo.data_ptr()
    _lib.call('sfgpi_step_prep', C.byref(pr), st)
    torch.cuda.synchronize()
    assert torch.equal(lib._shadow_for('online').view(torch.int16), ref_on.view(torch.int16))
    assert torch.equal(lib._shadow_for('target').view(torch.int16), ref_tg.view(torch.int16))
    assert torch.equal(keys, keys_ref) and int(keys.view(-1)[-1]) == 0          # the element past n_keys is untouched
    assert torch.equal(wq.view(torch.int16), wq_ref.view(torch.int16)) and torch.equal(bq, bq_ref)
    assert torch.equal(xo.view(torch.int16), xo_ref.view(torch.int16))


@pytest.mark.parametrize('kind', ['pinned', 'pageable'])
def test_train_step_from_host_batches_equals_device_batches(kind):
    """Host-resident replay batches (pinned: pulled over PCIe by the prologue kernel itself; pageable: cudaMemcpyAsync
    commands) must give bit-identical steps to device-resident batches."""
    S, A, D, N, B = 4, 9, 12, 3, 1000
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N, gdim=100, beta=1, use_gpi=True)
    o, gen = make(S, A, D, N, seed=41, tsf_dim=100)
    batches = [synthetic_transitions(B, S, A, D, gen) for _ in range(3)]
    sf_d, ag_d = gu.build_g3(meta, oracle=o)
    sf_h, ag_h = gu.build_g3(meta, oracle=o)
    sf_d._library.set_precision('bf16')
    sf_h._library.set_precision('bf16')
    for tr in batches:
        host = tuple(t.pin_memory() for t in tr) if kind == 'pinned' else tr
        ld = ag_d.update_successor_all(tuple(t.cuda() for t in tr), use_gpi=True)
        lh = ag_h.update_successor_all(host, use_gpi=True)
        torch.cuda.synchronize()
        assert torch.equal(ld, lh)
    n = N
    assert torch.equal(sf_d._library.online[:n], sf_h._library.online[:n])
    assert torch.equal(sf_d._library.g[:n], sf_h._library.g[:n]) and torch.equal(sf_d._library.h, sf_h._library.h)
    # asynchronous read-back of the losses as the last command of the step
    hl = torch.zeros(N, 3).pin_memory() if kind == 'pinned' else torch.zeros(N, 3)
    ld = ag_d.update_successor_all(tuple(t.cuda() for t in batches[0]), use_gpi=True, host_losses=hl)
    torch.cuda.current_stream().synchronize()
    assert torch.equal(hl, ld.cpu()) and float(hl.abs().sum()) > 0
    ld2 = ag_d.update_successor_all(tuple(t.cuda() for t in batches[1]), use_gpi=True)      # and the slot switches off again
    torch.cuda.synchronize()
    assert not torch.equal(hl, ld2.cpu())


@pytest.mark.parametrize('S,A,D,N,B,nws', [(4, 9, 12, 3, 1000, (4, 5, 8, 13, 40)), (11, 27, 50, 2, 333, (6, 10)), (4, 2, 20, 2, 200, (4, 9, 70))])
def test_multi_vector_gpi_keys_equal_single_vector_runs(S, A, D, N, B, nws):
    """
    The folded GPI output layer interleaves reward vectors in blocks of 8 (4) columns (csrc/mlp_forward_tc.cu: gpi_wblock).
    Every output element is an independent dot product, so scoring n_w vectors in one launch must give, for every vector,
    exactly the keys of a single-vector launch -- across block padding, 256-column chunk boundaries and ragged row tiles.
    """
    import ctypes as C
    from deep_successor_features_for_transfer_b200 import _lib
    from deep_successor_features_for_transfer_b200.library import _stream
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make(S, A, D, N, seed=47)
    sf = gu.build_g2(meta, oracle=o, hyper=HYPER_BF16)
    lib = sf._library
    x = synthetic_transitions(B, S, A, D, gen)[0].cuda()
    lib._pack('online', 0, N)

    def run(w):
        nw = w.shape[0]
        ka = torch.empty(nw, B, dtype=torch.int64, device='cuda')
        kt = torch.empty(nw, B, dtype=torch.int64, device='cuda')
        _lib.call('sfgpi_keys_fill', ka.data_ptr(), ka.numel(), _stream())
        _lib.call('sfgpi_keys_fill', kt.data_ptr(), kt.numel(), _stream())
        a = lib._fwd_args(lib.online, 0, N, x)
        a.w, a.n_w, a.w_diag, a.task_base = w.data_ptr(), nw, 0, 7
        a.key_action, a.key_task = ka.data_ptr(), kt.data_ptr()
        q = torch.zeros(B, N, A, device='cuda')
        a.q_out = q.data_ptr()
        wq = torch.empty(N * _lib.lib().sfgpi_gpi_fold_rows(C.byref(lib.spec.desc()), nw) * 256, dtype=torch.bfloat16, device='cuda')
        bq = torch.empty(wq.numel() // 256, device='cuda')
        _lib.call('sfgpi_fold_gpi', C.byref(lib.spec.desc()), lib.online.data_ptr(), 0, N, w.data_ptr(), nw, 0, wq.data_ptr(), bq.data_ptr(), _stream())
        _lib.call('sfgpi_mlp_forward_tc', C.byref(a), lib._shadow_for('online').data_ptr(), lib.cap, wq.data_ptr(), bq.data_ptr(), _stream())
        torch.cuda.synchronize()
        return ka, kt, q

    for nw in nws:
        w = (torch.rand(nw, D, generator=gen) * 0.02 - 0.01).cuda().contiguous()
        ka, kt, q = run(w)
        for wi in sorted({0, 1, nw // 2, nw - 2, nw - 1}):
            ka1, kt1, q1 = run(w[wi:wi + 1].contiguous())
            assert torch.equal(ka[wi], ka1[0]) and torch.equal(kt[wi], kt1[0]), f'n_w={nw}, vector {wi}'
            if wi == 0:
                assert torch.equal(q, q1)                     # q_out carries reward vector 0
        # and the keys are the argmax of that q (vector 0), first-index ties
        assert torch.equal(lib.decode_keys(ka[0]), torch.argmax(q.max(dim=1).values, dim=-1))
        assert torch.equal(lib.decode_keys(kt[0]) - 7, torch.argmax(q.max(dim=2).values, dim=1))


# ------------------------------------------------------------------------------------------------------------------------
# K-step parity of the tensor-core TRAIN STEP (the path every BENCH / SCALE number comes from): post-step weights, Adam
# moments and losses of the all-task step after K = 1 and K = 10 steps, against
#   (a) the oracle with the kernels' own rounding points (oracle/sf_oracle.py: emulate='bf16' -- operands of every GEMM,
#       forward and backward, rounded to bf16, fp32 accumulation).  What is left is summation order plus the occasional value
#       that lands on the other side of a bf16 rounding boundary: bound EMUL_*;
#   (b) the reference's fp32 arithmetic: the mode's stated tolerance, bound FP32_*.
# Metrics: relative Frobenius error of the Adam first moment m (after one step m = 0.1 g: the gradient itself), of sqrt(v), and
# of the weight UPDATE W_K - W_0 (Adam's first steps move every weight by ~lr * sign(g), so a flipped sign of a noise-level
# gradient element is a full 2*lr error in that element: the update error is ~2 sqrt(fraction of flipped signs) and is the
# loosest of the three by construction).  The bounds are ~3x the values measured on B200 (profiles/r02_bf16_drift.md).
# ------------------------------------------------------------------------------------------------------------------------
# bounds[K] = (m, sqrt(v), dW, losses, fp32 side paths w / g / h): ~3x the worst value measured on B200 over the four cases
# (profiles/r02_bf16_drift.md).  K = 1 against the emulating oracle is the kernels' own error (5e-4 .. 8e-4 measured); the K = 10
# rows are trajectory divergence: Adam's early steps are ~lr * sign(g), so operand-rounding noise on near-zero gradient elements
# turns into full-size weight differences that feed the next step's forward.
EMUL = {1: dict(m=2.5e-3, v=2.5e-3, dw=3e-2, loss=1e-5, side=1e-5), 10: dict(m=0.12, v=0.045, dw=0.17, loss=4e-3, side=2.5e-3)}
FP32 = {1: dict(m=9e-2, v=9e-2, dw=0.6, loss=1e-3, side=6e-2), 10: dict(m=0.2, v=0.09, dw=0.36, loss=4e-3, side=6e-2)}


def _adam_views(lib, i):
    sp = lib.spec
    return sp.views(lib.m[i].cpu()), sp.views(lib.v[i].cpu())


def kstep_metrics(variant, N, K, B=4096, seed=51, precision='bf16'):
    """Runs K all-task steps on the CUDA path and on both oracles from identical weights / batches; returns worst-case metrics."""
    S, A, D = 4, 9, 12
    tsf = variant == 'g3'
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N, gdim=100, beta=1, use_gpi=True)
    o32, gen = make(S, A, D, N, seed=seed, tsf_dim=100 if tsf else None)
    oem, _ = make(S, A, D, N, seed=seed, tsf_dim=100 if tsf else None)
    oem.emulate = 'bf16' if precision == 'bf16' else ('tf32' if precision == 'tf32' else None)
    if tsf:
        sf, ag = gu.build_g3(meta, oracle=o32)
        sf._library.set_precision(precision)
    else:
        sf = ag = gu.build_g2(meta, oracle=o32, hyper=dict(gu.HYPER, precision=precision))
    lib = sf._library
    W0 = [[W.clone() for W, _ in o32.psi[i]] for i in range(N)]
    out = dict(emul=dict(m=0.0, v=0.0, dw=0.0, loss=0.0, w=0.0, g=0.0, h=0.0), fp32=dict(m=0.0, v=0.0, dw=0.0, loss=0.0, w=0.0, g=0.0, h=0.0))
    for k in range(K):
        tr = synthetic_transitions(B, S, A, D, gen)
        got = ag.update_successor_all(gu.cuda_tr(tr), use_gpi=True).cpu()
        for name, o in (('emul', oem), ('fp32', o32)):
            ref = o.ensemble_update_frozen(tr, tsf=tsf, use_gpi=True)
            for i in range(N):
                r = torch.stack([torch.as_tensor(float(x)) for x in ref[i]])
                out[name]['loss'] = max(out[name]['loss'], float(((got[i] - r).abs() / r.abs().clamp_min(1e-12)).max()))
    for name, o in (('emul', oem), ('fp32', o32)):
        for i in range(N):
            ms, vs = _adam_views(lib, i)
            params = gu.psi_params(sf, i)
            for l in range(len(params)):
                m_ref, v_ref = o.adam[i]['m']['sf'][2 * l], o.adam[i]['v']['sf'][2 * l]
                out[name]['m'] = max(out[name]['m'], fro_err(ms[l][0], m_ref))
                out[name]['v'] = max(out[name]['v'], fro_err(vs[l][0].sqrt(), v_ref.sqrt()))
                out[name]['dw'] = max(out[name]['dw'], fro_err(params[l][0] - W0[i][l], o.psi[i][l][0] - W0[i][l]))
            fw = sf.fit_w[i].weight.data.cpu()
            out[name]['w'] = max(out[name]['w'], rel_err(fw, o.w[i]))
            if tsf:
                out[name]['g'] = max(out[name]['g'], rel_err(ag.g_functions[i].weight.data.cpu(), o.g[i][0]))
        if tsf:
            out[name]['h'] = rel_err(ag.h_function.weight.data.cpu(), o.h[0])
        assert [int(s) for s in lib.step[:N].cpu()] == [o.adam[i]['step'] for i in range(N)]
    return out


@pytest.mark.parametrize('variant,N,K', [('g2', 4, 1), ('g3', 4, 1), ('g3', 4, 10), ('g2', 3, 10)])
def test_bf16_k_steps_weights_moments_losses(variant, N, K):
    mt = kstep_metrics(variant, N, K)
    e, f = mt['emul'], mt['fp32']
    msg = f'{variant} N={N} K={K}: {mt}'
    for got, bound in ((e, EMUL[K]), (f, FP32[K])):
        assert got['m'] < bound['m'] and got['v'] < bound['v'] and got['dw'] < bound['dw'] and got['loss'] < bound['loss'], msg
        # the fp32 side paths (reward head w, TSF g / h) see the operand rounding only through psi
        assert max(got['w'], got['g'], got['h']) < bound['side'], msg


def test_bf16_1001_steps_cross_a_target_sync():
    """
    SURVEY 8c: K = 1001 single-policy TSF steps crossing the target sync at update 1000 (target_update_ev = 1000), bf16 mode
    against the fp32 oracle on the same 16 recycled batches (B = 256, 2 policies).  Stated drift bound on the 1001 (loss, l1,
    l2) triples relative to the fp32 trajectory: first 100 steps < 1.5e-2, median < 3e-2, every step < 0.3.  Measured on B200
    (profiles/r02_bf16_drift.md): 4.2e-3 / 8.9e-3 / 0.108 -- and the oracle with bf16-rounded operands drifts from the fp32
    oracle by 6.5e-3 / 9.8e-3 / 0.149 on the same run, i.e. the late-run drift is the mode's rounding amplified by 1000 Adam
    steps on 16 recycled batches, not kernel error.  After the run the target net is the online net of update 1000 (one
    further update applied to online only), the sync counter restarted.
    """
    LOSS_DRIFT_100, LOSS_DRIFT_MEDIAN, LOSS_DRIFT_MAX = 1.5e-2, 3e-2, 0.3
    S, A, D, N, B, K = 4, 9, 12, 2, 256, 1001
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N, gdim=100, beta=1, use_gpi=True, target_update_ev=1000)
    o, gen = make(S, A, D, N, seed=61, tsf_dim=100)
    o.target_update_ev = 1000
    sf, ag = gu.build_g3(meta, oracle=o)
    sf._library.set_precision('bf16')
    batches = [synthetic_transitions(B, S, A, D, gen) for _ in range(16)]
    dev_b = [gu.cuda_tr(b) for b in batches]
    got, ref = [], []
    tgt_before = gu.psi_params(sf, 1, target=True)[1][0].clone()
    for k in range(K):
        got.append(torch.stack(list(ag.update_successor(dev_b[k % 16], 1, True))))
        ref.append([float(x) for x in o.tsf_update_successor(batches[k % 16], 1, True)])
        if k == 999:
            online_at_sync = [W.clone() for W, _ in gu.psi_params(sf, 1)]
    got = torch.stack(got).cpu().double().numpy()
    ref = np.array(ref)
    drift = np.abs(got - ref) / np.maximum(np.abs(ref), 1e-9)
    assert drift.max() < LOSS_DRIFT_MAX, f'worst loss drift {drift.max():.3e} at step {int(drift.max(axis=1).argmax())}'
    assert float(np.median(drift)) < LOSS_DRIFT_MEDIAN and drift[:100].max() < LOSS_DRIFT_100, (float(np.median(drift)), drift[:100].max())
    assert sf.updates_since_target_updated[1] == 1 and o.updates_since_target_updated[1] == 1
    tgt = [W for W, _ in gu.psi_params(sf, 1, target=True)]
    assert all(torch.equal(a, b) for a, b in zip(tgt, online_at_sync))          # target == online of update 1000, bit for bit
    assert not torch.equal(tgt[1], tgt_before)
    assert not torch.equal(tgt[1], gu.psi_params(sf, 1)[1][0])                    # ... and online has moved on since


def test_bf16_gpi_256_reward_vectors_vs_oracle():
    """
    BASELINE config 4's GPI epilogue (n_w = 256 reward vectors, 2304 folded output columns = 9 chunks of 256, blocked column
    order) against the ORACLE, not against itself: for every one of the 256 vectors the action key must be the oracle's
    argmax_a max_j q (ties inside the bf16 tolerance may flip) and the key's value within BF16_TOL of the oracle's max.
    """
    import ctypes as C
    from deep_successor_features_for_transfer_b200 import _lib
    from deep_successor_features_for_transfer_b200.library import _stream
    S, A, D, N, B, NW = 4, 9, 12, 6, 700, 256
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make(S, A, D, N, seed=71)
    sf = gu.build_g2(meta, oracle=o, hyper=HYPER_BF16)
    lib = sf._library
    x = synthetic_transitions(B, S, A, D, gen)[0]
    w = (torch.rand(NW, D, generator=gen) * 0.02 - 0.01).contiguous()
    lib._pack('online', 0, N)
    ka = torch.empty(NW, B, dtype=torch.int64, device='cuda')
    kt = torch.empty(NW, B, dtype=torch.int64, device='cuda')
    _lib.call('sfgpi_keys_fill', ka.data_ptr(), ka.numel(), _stream())
    _lib.call('sfgpi_keys_fill', kt.data_ptr(), kt.numel(), _stream())
    xd, wd = x.cuda(), w.cuda()
    a = lib._fwd_args(lib.online, 0, N, xd)
    a.w, a.n_w, a.w_diag, a.task_base = wd.data_ptr(), NW, 0, 0
    a.key_action, a.key_task = ka.data_ptr(), kt.data_ptr()
    wq, bq = lib._fold(a, 'online')
    _lib.call('sfgpi_mlp_forward_tc', C.byref(a), lib._shadow_for('online').data_ptr(), lib.cap, wq.data_ptr(), bq.data_ptr(), _stream())
    torch.cuda.synchronize()
    act, val = lib.decode_keys(ka, want_value=True)
    task = lib.decode_keys(kt)
    psi = o.get_successors(x)                                                     # [B,N,A,D] fp32 oracle
    q_all = torch.einsum('bnad,wd->wbna', psi, w)                                 # [NW,B,N,A]
    scale = float(q_all.abs().max())
    n_flip = 0
    for wi in range(NW):
        q = q_all[wi]
        assert float((val[wi].cpu() - q.reshape(B, -1).max(dim=1).values).abs().max()) < BF16_TOL * scale
        a_ref = torch.argmax(q.max(dim=1).values, dim=-1)
        t_ref = torch.argmax(q.max(dim=2).values, dim=1)
        ok, nb = gu.argmax_mismatch_ok(q, a_ref, act[wi].cpu(), 'action', BF16_TOL)
        assert ok, f'vector {wi}: {nb} action mismatches outside tolerance'
        ok2, nb2 = gu.argmax_mismatch_ok(q, t_ref, task[wi].cpu(), 'task', BF16_TOL)
        assert ok2, f'vector {wi}: {nb2} task mismatches outside tolerance'
        n_flip += nb
    assert n_flip < 0.03 * NW * B                                                 # flips are confined to near-ties (SURVEY 7: ~0.5 %)


def test_bf16_ensemble_step_32_policies_vs_frozen_oracle():
    """The multi-vector train step at n_w = N = 32 (the 8-GPU shard's GPI width) against the frozen-snapshot oracle, B = 256."""
    S, A, D, N, B = 4, 9, 12, 32, 256
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N, gdim=100, beta=30, use_gpi=True)
    o, gen = make(S, A, D, N, seed=73, tsf_dim=100, beta=30)
    sf, ag = gu.build_g3(meta, oracle=o)
    sf._library.set_precision('bf16')
    tr = synthetic_transitions(B, S, A, D, gen)
    ref = o.ensemble_update_frozen(tr, tsf=True, use_gpi=True)
    got = ag.update_successor_all(gu.cuda_tr(tr), use_gpi=True).cpu()
    for i in range(N):
        assert np.allclose(got[i].numpy(), [float(v) for v in ref[i]], rtol=3e-2, atol=1e-6), (i, got[i], ref[i])
    assert rel_err(ag.h_function.weight.data.cpu(), o.h[0]) < 2e-2


def test_bf16_hopper_64_policies_65536_states_spot_check_vs_oracle():
    """
    BASELINE config 3 at FULL size (Hopper S11/A27/D50, 64 policies, 65 536 states, bf16 mode): the fused GPI keys of 512 spot
    states against the fp32 oracle's GPI over all 64 policies -- value within BF16_TOL, action / task equal except ties inside
    the tolerance -- plus size-independent properties over all 65 536 states (indices in range, key value == max of q_out rows).
    """
    S, A, D, N, B = 11, 27, 50, 64, 65536
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make(S, A, D, N, seed=79)
    sf = gu.build_g2(meta, oracle=o, hyper=HYPER_BF16)
    lib = sf._library
    x = torch.sigmoid(torch.randn(B, S, generator=gen))
    w = sf.fit_w[5].weight.data.cpu().reshape(-1)
    q_dev, ka, kt = lib.gpi(x.cuda(), w, want_q=True)
    act, val = lib.decode_keys(ka, want_value=True)
    task = lib.decode_keys(kt)
    assert int(act.min()) >= 0 and int(act.max()) < A and int(task.min()) >= 0 and int(task.max()) < N
    assert torch.equal(val, q_dev.reshape(B, -1).max(dim=1).values)
    spot = torch.arange(0, B, B // 512)[:512]
    q_ref, task_ref = o.GPI_w(x[spot], w)
    scale = float(q_ref.abs().max())
    assert float((val[spot.cuda()].cpu() - q_ref.reshape(512, -1).max(dim=1).values).abs().max()) < BF16_TOL * scale
    a_ref = torch.argmax(q_ref.max(dim=1).values, dim=-1)
    ok, nb = gu.argmax_mismatch_ok(q_ref, a_ref, act[spot.cuda()].cpu(), 'action', BF16_TOL)
    assert ok, f'{nb} action mismatches outside tolerance'
    ok, nb = gu.argmax_mismatch_ok(q_ref, task_ref, task[spot.cuda()].cpu(), 'task', BF16_TOL)
    assert ok, f'{nb} task mismatches outside tolerance'


@pytest.mark.parametrize('NW,B', [(256, 700), (77, 300), (64, 1000), (16, 257)])
def test_bf16_gpi_wide_scan_equals_rolled_scan(NW, B):
    """
    The scan for many reward vectors (gpi_scan_wide8, csrc/forward_tc.cuh: 32-column windows, prefetched TMEM loads, lean
    emission) must leave exactly the keys of the rolled 8-column scan: action and task keys, vector counts that are not a
    multiple of 8, ragged row tiles, ranges that end inside a 32-column window (the rest goes through the rolled scan).
    """
    import ctypes as C
    from deep_successor_features_for_transfer_b200 import _lib
    from deep_successor_features_for_transfer_b200.library import _stream
    S, A, D, N = 4, 9, 12, 3
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make(S, A, D, N, seed=73)
    sf = gu.build_g2(meta, oracle=o, hyper=HYPER_BF16)
    lib = sf._library
    xd = synthetic_transitions(B, S, A, D, gen)[0].cuda()
    wd = (torch.rand(NW, D, generator=gen) * 0.02 - 0.01).cuda().contiguous()
    lib._pack('online', 0, N)

    def run(wide_min):
        ka = torch.empty(NW, B, dtype=torch.int64, device='cuda')
        kt = torch.empty(NW, B, dtype=torch.int64, device='cuda')
        _lib.call('sfgpi_keys_fill', ka.data_ptr(), ka.numel(), _stream())
        _lib.call('sfgpi_keys_fill', kt.data_ptr(), kt.numel(), _stream())
        a = lib._fwd_args(lib.online, 0, N, xd)
        a.w, a.n_w, a.w_diag, a.task_base = wd.data_ptr(), NW, 0, 5
        a.key_action, a.key_task = ka.data_ptr(), kt.data_ptr()
        wq, bq = lib._fold(a, 'online')
        old_c = _lib.lib().sfgpi_set_option(b'forward_chain', 0)            # the ping-pong pair kernel (the one large launches take)
        old_w = _lib.lib().sfgpi_set_option(b'gpi_wide_min', wide_min)
        try:
            _lib.call('sfgpi_mlp_forward_tc', C.byref(a), lib._shadow_for('online').data_ptr(), lib.cap, wq.data_ptr(), bq.data_ptr(), _stream())
            torch.cuda.synchronize()
        finally:
            _lib.lib().sfgpi_set_option(b'forward_chain', old_c)
            _lib.lib().sfgpi_set_option(b'gpi_wide_min', old_w)
        return ka, kt

    ka_w, kt_w = run(0)
    ka_r, kt_r = run(1 << 30)
    assert torch.equal(ka_w, ka_r) and torch.equal(kt_w, kt_r)
    assert int((ka_w == torch.iinfo(torch.int64).min).sum()) == 0


@pytest.mark.parametrize('S,A,D,N,NW', [(4, 9, 12, 3, 256), (4, 9, 12, 9, 77), (11, 27, 50, 4, 40)])
def test_large_gpi_fold_by_units_equals_row_by_row(S, A, D, N, NW):
    """
    Folds of >= 4096 rows run one block per (policy, action, block-of-vectors) unit (csrc/mlp_forward_tc.cu: fold_unit; inside a
    train step as the prologue's second launch), smaller ones one block per folded row.  Same fmaf chain per output: the
    all-policies fold (by units) must equal the policy-by-policy folds (row by row) bit for bit -- D <= 16 (rows in
    registers) and D = 50 (rows from L1), vector counts that pad the last block, and sfgpi_step_prep's two-launch form.
    """
    import ctypes as C
    from deep_successor_features_for_transfer_b200 import _lib
    from deep_successor_features_for_transfer_b200.library import _stream
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N)
    o, gen = make(S, A, D, N, seed=77)
    sf = gu.build_g2(meta, oracle=o, hyper=HYPER_BF16)
    lib = sf._library
    desc = lib.spec.desc()
    st = _stream()
    w = (torch.rand(NW, D, generator=gen) * 0.02 - 0.01).cuda().contiguous()
    nq = _lib.lib().sfgpi_gpi_fold_rows(C.byref(desc), NW)
    assert nq * N >= 4096 > nq
    wq = torch.full((N, nq, 256), 7.0, dtype=torch.bfloat16, device='cuda')
    bq = torch.full((N, nq), 7.0, device='cuda')
    _lib.call('sfgpi_fold_gpi', C.byref(desc), lib.online.data_ptr(), 0, N, w.data_ptr(), NW, 0, wq.data_ptr(), bq.data_ptr(), st)
    wq1 = torch.full((N, nq, 256), 3.0, dtype=torch.bfloat16, device='cuda')
    bq1 = torch.full((N, nq), 3.0, device='cuda')
    for i in range(N):
        _lib.call('sfgpi_fold_gpi', C.byref(desc), lib.online.data_ptr(), i, 1, w.data_ptr(), NW, 0, wq1[i].data_ptr(), bq1[i].data_ptr(), st)
    torch.cuda.synchronize()
    assert torch.equal(wq.view(torch.int16), wq1.view(torch.int16)) and torch.equal(bq, bq1)
    assert float(wq.float().abs().sum()) > 0
    # the same fold as the second launch of the step prologue
    pr = _lib.StepPrepArgs()
    pr.net = desc
    pr.fold_params, pr.fold_lo, pr.fold_n = lib.online.data_ptr(), 0, N
    wq2, bq2 = torch.zeros_like(wq), torch.zeros_like(bq)
    pr.w, pr.n_w, pr.w_diag, pr.wq, pr.bq = w.data_ptr(), NW, 0, wq2.data_ptr(), bq2.data_ptr()
    assert _lib.lib().sfgpi_step_prep_launches(C.addressof(pr)) == 2
    _lib.call('sfgpi_step_prep', C.byref(pr), st)
    torch.cuda.synchronize()
    assert torch.equal(wq2.view(torch.int16), wq.view(torch.int16)) and torch.equal(bq2, bq)


def test_adam_losses_host_needs_pinned_memory():
    """sfgpi_adam_args.losses_host: pinned host memory is written by the kernel; pageable memory is refused, loudly."""
    import ctypes as C
    from deep_successor_features_for_transfer_b200 import _lib
    S, A, D, N, B = 4, 9, 12, 2, 256
    meta = dict(S=S, A=A, D=D, hidden=[256, 256], acts=['relu', 'relu'], N=N, gdim=100, beta=1, use_gpi=True)
    o, gen = make(S, A, D, N, seed=79, tsf_dim=100)
    sf, ag = gu.build_g3(meta, oracle=o)
    sf._library.set_precision('bf16')
    tr = gu.cuda_tr(synthetic_transitions(B, S, A, D, gen))
    hl = torch.zeros(N, 3).pin_memory()
    got = ag.update_successor_all(tr, use_gpi=True, host_losses=hl)
    torch.cuda.synchronize()
    assert torch.equal(hl, got.cpu()) and float(hl.abs().sum()) > 0
    lib = sf._library
    ad = lib._ws[lib.last_plan_key]['ad']
    pageable = torch.zeros(N, 3)
    ad.losses_host = pageable.data_ptr()
    rc = _lib.lib().sfgpi_adam_step(C.byref(ad), None)
    assert rc != 0 and b'pinned' in _lib.lib().sfgpi_last_error()
    ad.losses_host = None
