"""
CPU-only tests (no compute calls): the C-ABI library loads and exports every symbol include/sfgpi.h declares, the ctypes
structs mirror the header field for field, and the multi-GPU host logic (shard ranges, packed (value,index) keys, MAX
all-reduce) behaves on a world_size-2 gloo group exactly like the single-process computation.
"""
import os
import re
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from deep_successor_features_for_transfer_b200 import _lib, dist as sdist
from tests import gpu_util as gu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, 'include', 'sfgpi.h')


def header_text():
    with open(HEADER) as f:
        return re.sub(r'/\*.*?\*/', '', f.read(), flags=re.S)


def test_library_exports_every_declared_symbol():
    declared = set(re.findall(r'\b(sfgpi_[a-z0-9_]+)\s*\(', header_text()))
    assert declared, 'no prototypes found in include/sfgpi.h'
    handle = _lib.lib()                              # builds with nvcc if the .so is missing; raises if it cannot
    for name in sorted(declared):
        assert hasattr(handle, name), f'libsfgpi.so does not export {name}'
    assert declared == set(_lib.SYMBOLS), f'binding/header mismatch: {declared ^ set(_lib.SYMBOLS)}'
    assert handle.sfgpi_version() >= 100
    assert isinstance(handle.sfgpi_last_error(), bytes)


def c_struct_fields(name):
    text = header_text()
    end = re.search(r'\}\s*' + name + r'\s*;', text)
    assert end, name
    body = text[text.rfind('typedef struct {', 0, end.start()) + len('typedef struct {'):end.start()]
    fields = []
    for decl in body.split(';'):
        decl = decl.strip()
        if not decl:
            continue
        decl = re.sub(r'^(const\s+)?[A-Za-z_0-9]+(\s+const)?\s*', '', decl, count=1)      # drop the base type
        for part in decl.split(','):
            fields.append(re.sub(r'[\*\s]|\[.*?\]', '', part))
    return fields


@pytest.mark.parametrize('cname,pyname', [('sfgpi_net_desc', 'NetDesc'), ('sfgpi_forward_args', 'ForwardArgs'),
                                          ('sfgpi_td_args', 'TdArgs'), ('sfgpi_backward_args', 'BackwardArgs'),
                                          ('sfgpi_backward_tc_args', 'BackwardTcArgs'), ('sfgpi_forward_tc_job', 'ForwardTcJob'), ('sfgpi_cmd', 'Cmd'), ('sfgpi_replay_args', 'ReplayArgs'),
                                          ('sfgpi_adam_segment', 'AdamSegment'), ('sfgpi_adam_args', 'AdamArgs'),
                                          ('sfgpi_step_prep_args', 'StepPrepArgs'), ('sfgpi_peer_ctx', 'PeerCtx'),
                                          ('sfgpi_peer_keys_args', 'PeerKeysArgs'), ('sfgpi_peer_unpack_args', 'PeerUnpackArgs')])
def test_ctypes_structs_mirror_header(cname, pyname):
    assert c_struct_fields(cname) == [f[0] for f in getattr(_lib, pyname)._fields_]


def test_negative_sizes_are_rejected_without_a_gpu():
    """Argument validation happens before any CUDA call, so it is testable here: rc < 0 and an error text."""
    a = _lib.ForwardArgs()
    a.net.n_layers = 0
    rc = _lib.lib().sfgpi_mlp_forward(a, None)
    assert rc < 0 and len(_lib.lib().sfgpi_last_error()) > 0


def test_new_entry_points_validate_before_touching_cuda():
    """sfgpi_step_prep / sfgpi_phi_head / peer exchange / sfgpi_adam_step: bad arguments -> rc < 0 with an error text, no CUDA call needed."""
    import ctypes as C
    L = _lib.lib()
    pr = _lib.StepPrepArgs()                                        # zeroed descriptor: not a tensor-core shape
    assert L.sfgpi_step_prep(C.byref(pr), None) < 0 and b'sfgpi_step_prep' in L.sfgpi_last_error()
    assert L.sfgpi_phi_head(None, None, None, 32, 20, None, None, None, None) < 0 and b'sfgpi_phi_head' in L.sfgpi_last_error()
    assert L.sfgpi_phi_head_partials(32) == 1 and L.sfgpi_phi_head_partials(300) == 2 and L.sfgpi_phi_head_partials(0) == 1
    ka = _lib.PeerKeysArgs()
    ka.ctx.world, ka.ctx.rank = 99, 0                               # more than SFGPI_MAX_PEERS
    assert L.sfgpi_peer_reduce_keys(C.byref(ka), None) < 0 and b'peers' in L.sfgpi_last_error()
    ua = _lib.PeerUnpackArgs()
    ua.ctx.world, ua.ctx.rank = 2, 0                                # flag blocks not mapped
    assert L.sfgpi_peer_unpack(C.byref(ua), None) < 0 and b'not mapped' in L.sfgpi_last_error()
    t = _lib.TdArgs()
    t.variant, t.B, t.n_pol, t.D, t.aux_len = 1, 8, 1, 4, 4
    ka2 = _lib.PeerKeysArgs()
    t.peer_keys = C.addressof(ka2)                                  # peer keys without next_psi / a valid context
    assert L.sfgpi_td_step(C.byref(t), None) < 0 and b'peer_keys' in L.sfgpi_last_error()
    assert _lib.MAX_PEERS == 16 and C.sizeof(_lib.Cmd) == 80
    # sfgpi_adam_step: a step that is not fresh reads `consts` and writes the next step's corrections into a distinct `consts_next`
    host = (C.c_double * 8)(), (C.c_double * 8)(), (C.c_int32 * 2)()
    ad = _lib.AdamArgs()
    ad.n_seg, ad.n_pol, ad.step = 1, 1, C.addressof(host[2])
    ad.seg[0].len, ad.seg[0].n_part = 4, 1
    for consts, consts_next, missing in ((None, C.addressof(host[1]), b'needs consts'), (C.addressof(host[0]), None, b'needs consts_next'),
                                         (C.addressof(host[0]), C.addressof(host[0]), b'distinct from consts')):
        ad.consts, ad.consts_next = consts, consts_next
        assert L.sfgpi_adam_step(C.byref(ad), None) < 0 and L.sfgpi_last_error().endswith(missing)


def test_bf16_shadow_and_fold_refuse_s64_like_the_backward():
    """The bf16 backward, the step prologue and the state gradient need S <= 63 (xo = [x | 1 | 0...] is 64 columns wide), so the
    bf16 pack and GPI fold -- the first calls a bf16 library makes -- refuse S = 64 up front instead of building a library
    whose every train step fails.  S = 63 passes validation (n_pol = 0: nothing is launched)."""
    import ctypes as C
    from deep_successor_features_for_transfer_b200.library import NetSpec
    L = _lib.lib()
    for S, ok in ((64, False), (63, True)):
        desc = NetSpec([S, 256, 256, 256, 108], ['none', 'relu', 'relu', 'none'], 9, 12).desc()
        n_pol = 0 if ok else 1                                      # S = 64 with one policy: refused before any pointer is read
        rc_pack = L.sfgpi_pack_bf16(C.byref(desc), None, 0, n_pol, None, None)
        err_pack = L.sfgpi_last_error()
        rc_fold = L.sfgpi_fold_gpi(C.byref(desc), None, 0, n_pol, None, 1, 0, None, None, None)
        err_fold = L.sfgpi_last_error()
        if ok:
            assert rc_pack == 0 and rc_fold == 0
        else:
            assert rc_pack == -1 and b'sfgpi_pack_bf16' in err_pack and b'S <= 63' in err_pack       # SFGPI_E_INVALID
            assert rc_fold == -1 and b'sfgpi_fold_gpi' in err_fold and b'S <= 63' in err_fold


def test_shard_range_partitions_exactly():
    for n_total in (1, 4, 7, 64, 256):
        for world in (1, 2, 3, 8):
            rng = [sdist.shard_range(n_total, world, r) for r in range(world)]
            assert rng[0][0] == 0 and rng[-1][1] == n_total
            assert all(rng[r][1] == rng[r + 1][0] for r in range(world - 1))
            sizes = [hi - lo for lo, hi in rng]
            assert max(sizes) - min(sizes) <= 1


def test_key_packing_orders_like_argmax_first_index():
    g = torch.Generator().manual_seed(3)
    q = torch.randn(257, 5, 9, generator=g)
    q[::7] = q[::7].round()                                         # force exact ties (and +-0)
    q[3, :, :] = 0.0
    q[4, 0, 0], q[4, 1, 0] = 0.0, -0.0
    ka, kt = sdist.gpi_keys_from_q(q)
    va, ia = sdist.unpack_keys(ka)
    vt, it = sdist.unpack_keys(kt)
    assert torch.equal(ia, torch.argmax(q.max(dim=1).values, dim=-1))          # sfdqn.py:316
    assert torch.equal(it, torch.argmax(q.max(dim=2).values, dim=-1))          # sfdqn.py:239
    assert torch.equal(va, q.reshape(257, -1).max(dim=1).values + 0.0) and torch.equal(va, vt)
    v, i = sdist.unpack_keys(sdist.pack_keys(torch.tensor([-1.5, 0.0, 2.0 ** 127, -2.0 ** 127]), torch.tensor([0, 7, 2 ** 31, 5])))
    assert v.tolist() == [-1.5, 0.0, 2.0 ** 127, -2.0 ** 127] and i.tolist() == [0, 7, 2 ** 31, 5]



def test_key_packing_never_selects_nan():
    """NaN is never selected, +-inf order as values, a row of NaN / -inf only decodes to index 0 (task: task_base), as on the
    device (tests/gpu_util.py::gpi_rule)."""
    g = torch.Generator().manual_seed(5)
    q = torch.randint(-2, 3, (64, 3, 9), generator=g).float()
    neg_nan = (torch.tensor(float('nan')).view(torch.int32) | -2 ** 31).view(torch.float32)
    q[0:8, :, 0] = float('nan')                                     # NaN first, beside finite maxima
    q[8:16] = float('nan')
    q[16:24] = neg_nan
    q[24:32] = float('-inf')
    q[32:40, 1, 2] = float('inf')
    q[32:36, 2, 1] = float('inf')
    q[40:48] = torch.where(torch.rand(8, 3, 9, generator=g) < 0.5, float('nan'), float('-inf'))
    q[48:56, :, 3:] = neg_nan
    q[56:64] = torch.where(torch.rand(8, 3, 9, generator=g) < 0.5, 0.0, -0.0)
    for task_base in (0, 5):
        ka, kt = sdist.gpi_keys_from_q(q, task_base=task_base)
        (va, ia), (vt, it) = sdist.unpack_keys(ka), sdist.unpack_keys(kt)
        cells = q.reshape(64, -1).double()
        a_ref, m = gu.gpi_rule(cells, torch.arange(9).repeat(3))
        t_ref, _ = gu.gpi_rule(cells, (task_base + torch.arange(3)).repeat_interleave(9))
        assert torch.equal(ia, a_ref) and torch.equal(it, t_ref)
        assert torch.equal(va.double(), m) and torch.equal(vt.double(), m)
        assert not va.isnan().any()
    assert int(ia[8]) == 0 and int(it[8]) == 5 and float(va[8]) == float('-inf')      # all NaN
    assert (int(ia[32]), int(it[32]), int(ia[36]), int(it[36])) == (1, 6, 2, 6)                 # ties at +inf

def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _gloo_worker(rank, world, port, q_all, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        n_total = q_all.shape[1]
        lo, hi = sdist.shard_range(n_total, world, rank)
        ctx = sdist.ShardContext(hi - lo)
        assert (ctx.lo, ctx.n_total, ctx.world, ctx.rank) == (lo, n_total, world, rank)
        ka, kt = sdist.gpi_keys_from_q(q_all[:, lo:hi], task_base=lo)           # this rank's policies only
        keys = torch.stack([ka, kt])
        sdist.allreduce_max_keys(keys)                                          # the one data-path collective
        if rank == 0:
            out.put(keys)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('n_total', [4, 5])
def test_sharded_gpi_equals_unsharded_gloo_world2(n_total):
    """Policies sharded over 2 ranks (even and uneven), keys MAX-all-reduced over gloo == single-process GPI."""
    g = torch.Generator().manual_seed(11)
    q = torch.randn(300, n_total, 9, generator=g)
    q[::5] = q[::5].round()                                       # ties across ranks must resolve to the smallest index
    ctx = mp.get_context('spawn')
    out = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q, out)) for r in range(2)]
    for p in procs:
        p.start()
    keys = out.get()
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    ka, kt = sdist.gpi_keys_from_q(q)
    assert torch.equal(keys[0], ka) and torch.equal(keys[1], kt)
    _, task = sdist.unpack_keys(keys[1])
    assert torch.equal(task, torch.argmax(q.max(dim=2).values, dim=-1))


# ---- host logic that needs no GPU ---------------------------------------------------------------------------------------
def test_no_cpu_fallback_constructors_raise_without_cuda():
    """The product has no CPU path: on a box without CUDA every public constructor fails loudly."""
    if torch.cuda.is_available():
        pytest.skip('needs a CUDA-less host')
    from deep_successor_features_for_transfer_b200.library import PackedSFLibrary
    from deep_successor_features_for_transfer_b200.sfdqn import DeepSF
    from deep_successor_features_for_transfer_b200.sfdqn_phi import PhiFunction
    from tests.gpu_util import FakeTask, model_lambda, HYPER
    with pytest.raises(RuntimeError, match='CUDA'):
        PackedSFLibrary()
    with pytest.raises(RuntimeError, match='CUDA'):
        sf = DeepSF(pytorch_model_handle=model_lambda([256, 256], ['relu', 'relu']), hyperparameters=dict(HYPER))
        sf.reset()
        sf.add_training_task(FakeTask(4, 9, 12, 0))
    with pytest.raises(RuntimeError, match='CUDA'):
        PhiFunction(4, 1, 20)


def test_missing_native_library_fails_loudly(tmp_path, monkeypatch):
    """No libsfgpi.so and no way to build it -> RuntimeError / OSError from _lib.lib(), never a silent fallback."""
    import deep_successor_features_for_transfer_b200._lib as L
    monkeypatch.setattr(L, '_lib', None)
    monkeypatch.setattr(L, 'LIB_PATH', str(tmp_path / 'libsfgpi_absent.so'))
    monkeypatch.setattr(L, 'CSRC', str(tmp_path))                     # no sources either: the build must fail
    (tmp_path / 'dummy.cuh').write_text('')
    with pytest.raises((RuntimeError, OSError)):
        L.lib()
    monkeypatch.undo()                                                # (restores the loaded handle and the real paths)
    assert L.lib().sfgpi_version() >= 100


def test_netspec_adopts_reference_shaped_models_and_rejects_the_rest():
    """utils/torch.py:19-22 shapes (Linear / ReLU / Tanh / Unflatten) are introspected; anything else is rejected."""
    from collections import OrderedDict
    from deep_successor_features_for_transfer_b200.library import NetSpec
    from tests.gpu_util import model_lambda
    model, _, _ = model_lambda([256, 256], ['relu', 'tanh'])(4, 9 * 12, (9, 12), 1)
    spec, linears = NetSpec.from_module(model, 9, 12)
    assert spec.dims == [4, 256, 256, 256, 108] and spec.acts == ['none', 'relu', 'tanh', 'none'] and len(linears) == 4
    assert spec.n_params == sum(p.numel() for p in model.parameters()) == 160620      # SURVEY 8: P(Reacher) = 160 620
    assert all(o % 4 == 0 for o in spec.w_off + spec.b_off) and spec.row_stride % 32 == 0 and spec.row_stride >= spec.n_params
    d = spec.desc()
    assert d.n_layers == 4 and list(d.dims)[:5] == spec.dims and d.n_actions == 9 and d.n_features == 12
    views = spec.views(torch.arange(spec.row_stride, dtype=torch.float32))
    assert [tuple(W.shape) for W, _ in views] == [(256, 4), (256, 256), (256, 256), (108, 256)]
    bad = torch.nn.Sequential(OrderedDict(a=torch.nn.Linear(4, 8), b=torch.nn.Sigmoid(), c=torch.nn.Linear(8, 108)))
    with pytest.raises(TypeError, match='unsupported layer'):
        NetSpec.from_module(bad, 9, 12)
    with pytest.raises(ValueError, match='n_actions \\* n_features'):
        NetSpec.from_module(model, 9, 13)
    with pytest.raises(ValueError, match='linear'):
        NetSpec.from_module(torch.nn.Sequential(torch.nn.Linear(4, 108), torch.nn.ReLU()), 9, 12)
    with pytest.raises(ValueError, match='bias'):
        NetSpec.from_module(torch.nn.Sequential(torch.nn.Linear(4, 108, bias=False)), 9, 12)


def test_host_side_size_helpers_of_the_abi():
    """The pure-host helpers callers size their buffers with (no CUDA call inside): values for the reference's shapes."""
    import ctypes as C
    from deep_successor_features_for_transfer_b200.library import NetSpec
    L = _lib.lib()

    def desc(S, A, D):
        dims = [S, 256, 256, 256, A * D]
        return NetSpec(dims, ['none', 'relu', 'relu', 'none'], A, D).desc()

    reacher, hopper, cartpole = desc(4, 9, 12), desc(11, 27, 50), desc(4, 2, 20)
    # bf16 shadow rows per policy: 3 x 256 (input + 2 hidden) + A*D padded to 16
    assert L.sfgpi_bf16_rows_per_policy(C.byref(reacher)) == 768 + 112
    assert L.sfgpi_bf16_rows_per_policy(C.byref(hopper)) == 768 + 1360
    assert L.sfgpi_bf16_rows_per_policy(C.byref(cartpole)) == 768 + 48
    # folded GPI rows: reward vectors in blocks of WB = 8 (4 for 4..7, 1 below), n_w padded to WB, x A, padded to 16
    fold = lambda d, nw: L.sfgpi_gpi_fold_rows(C.byref(d), nw)
    assert fold(reacher, 1) == 16 and fold(reacher, 3) == 32                  # plain order: n_w * 9 -> 16
    assert fold(reacher, 4) == 48 and fold(reacher, 5) == 80                  # WB = 4: 36 -> 48; 5 -> 8 vectors: 72 -> 80
    assert fold(reacher, 8) == 80 and fold(reacher, 32) == 288 and fold(reacher, 256) == 2304
    assert fold(hopper, 1) == 32 and fold(hopper, 10) == 432                 # 27 -> 32; 10 -> 16 vectors x 27
    for nw in range(1, 70):                                                   # never fewer rows than real (vector, action) pairs
        assert fold(reacher, nw) >= nw * 9 and fold(reacher, nw) % 16 == 0
    # TD partials: one per 8-CTA cluster of 32-row CTAs; phi-head partials: one per 256 rows
    assert [L.sfgpi_td_partials(b) for b in (0, 1, 256, 257, 4096)] == [1, 1, 1, 2, 16]
    assert [L.sfgpi_phi_head_partials(b) for b in (1, 256, 257)] == [1, 1, 2]
    # wgrad split-K: splits of whole 64-row groups, none empty
    for B in (32, 1000, 4096, 4219, 65536):
        for want in (1, 3, 5, 8, 64):
            n = L.sfgpi_bwd_tc_splits(B, want)
            bs = (((B + want - 1) // want) + 63) // 64 * 64
            assert 1 <= n <= want and (n - 1) * bs < B <= n * bs and L.sfgpi_bwd_tc_splits(B, n) == n
    assert L.sfgpi_bwd_tc_out_pad(C.byref(reacher)) >= 108 and L.sfgpi_bwd_tc_out_pad(C.byref(reacher)) % 64 == 0


def test_planar_flow_module_matches_the_oracle_on_cpu():
    """tsfdqn_nf's host surface (PlanarFlow, build_planar_flow; tsfdqn_nf.py:331-358): registered parameters in the reference's
    order, same forward as the oracle's g_apply."""
    import torch
    from deep_successor_features_for_transfer_b200 import tsfdqn_nf
    from oracle.sf_oracle import g_apply
    torch.manual_seed(3)
    g = tsfdqn_nf.PlanarFlow.build_planar_flow(4, 100, 5)
    assert [n for n, _ in g.named_parameters()][:3] == ['0.weight', '0.bias', '0.scale'] and len(list(g.parameters())) == 17
    assert all(float(p.abs().max()) <= 0.01 for f in list(g)[:-1] for p in f.parameters())
    x = torch.randn(7, 4)
    spec = [(f.weight.data, f.bias.data, f.scale.data) for f in list(g)[:-1]] + [(g[-1].weight.data, g[-1].bias.data)]
    assert torch.allclose(g(x), g_apply(x, spec), atol=1e-6)
    assert issubclass(tsfdqn_nf.TSFDQN, __import__('deep_successor_features_for_transfer_b200.tsfdqn', fromlist=['TSFDQN']).TSFDQN)
    assert tsfdqn_nf.DeepTSF is not None and tsfdqn_nf.ReplayBuffer is not None


def test_step_prep_launch_count_follows_the_fold_size():
    """sfgpi_step_prep_launches: folds of >= 4096 folded rows go out as the prologue's second launch (host logic, no GPU)."""
    import ctypes as C
    from deep_successor_features_for_transfer_b200.library import NetSpec
    spec = NetSpec([4, 256, 256, 256, 108], ['none', 'relu', 'relu', 'none'], 9, 12)
    pr = _lib.StepPrepArgs()
    pr.net = spec.desc()
    L = _lib.lib()
    assert L.sfgpi_step_prep_launches(C.addressof(pr)) == 1                       # no fold at all
    for n_pol, n_w, expect in ((4, 4, 1), (256, 256, 2), (1, 256, 1), (2, 256, 2), (52, 8, 2), (51, 8, 1)):
        pr.fold_n, pr.n_w, pr.w_diag = n_pol, n_w, 0
        rows = L.sfgpi_gpi_fold_rows(C.byref(pr.net), n_w)
        assert (rows * n_pol >= 4096) == (expect == 2)
        assert L.sfgpi_step_prep_launches(C.addressof(pr)) == expect, (n_pol, n_w)
    pr.fold_n, pr.n_w, pr.w_diag = 256, 256, 1                                    # diagonal: one vector per policy, 16 rows each
    assert L.sfgpi_step_prep_launches(C.addressof(pr)) == 2
