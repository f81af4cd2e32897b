# -*- coding: UTF-8 -*-
"""
ctypes binding of libsfgpi.so (C ABI declared in include/sfgpi.h).  There is NO fallback: if the shared library is missing
and cannot be built, or a call returns non-zero, a RuntimeError is raised.
"""
import ctypes as C
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB_PATH = os.environ.get('SFGPI_LIB_PATH') or os.path.join(HERE, 'libsfgpi.so')      # (override: A/B runs of two builds)
SOURCES = ['mlp_forward.cu', 'gpi.cu', 'td.cu', 'mlp_backward.cu', 'adam.cu', 'mlp_forward_tc.cu', 'mlp_chain_tc.cu', 'mlp_backward_tc.cu', 'run.cu', 'replay.cu', 'peer.cu', 'phi.cu', 'mlp_stream_tc.cu', 'mlp_wgrad_tf32.cu', 'g4.cu', 'target.cu', 'input_grad.cu']
MAX_LAYERS = 8
MAX_SEGMENTS = 8
ACT = {'none': 0, 'relu': 1, 'tanh': 2}
PREC = {'fp32': 0, 'bf16': 1, 'tf32': 2, 'tf32x3': 3}


def nvcc_path():
    """nvcc on PATH, else the one of the CUDA toolkit torch locates (CUDA_HOME / CUDA_PATH, /usr/local/cuda)."""
    found = shutil.which('nvcc')
    if found:
        return found
    from torch.utils.cpp_extension import CUDA_HOME
    if CUDA_HOME and os.path.isfile(os.path.join(CUDA_HOME, 'bin', 'nvcc')):
        return os.path.join(CUDA_HOME, 'bin', 'nvcc')
    raise RuntimeError('nvcc not found: put the CUDA toolkit\'s bin directory on PATH or set CUDA_HOME')


def build(force=False, verbose=False):
    """nvcc -> libsfgpi.so, sm_100a only (cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    deps = srcs + [os.path.join(CSRC, 'common.cuh'), os.path.join(HERE, '..', 'include', 'sfgpi.h')]
    deps += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith('.cuh')]
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(d) for d in deps):
        return LIB_PATH
    cmd = [nvcc_path(), '-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17', '-Xcompiler', '-fPIC',
           '-shared', '-o', LIB_PATH] + srcs
    if verbose:
        cmd.insert(1, '-Xptxas=-v')
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('nvcc failed building libsfgpi.so:\n' + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return LIB_PATH


class NetDesc(C.Structure):
    _fields_ = [('n_layers', C.c_int32), ('dims', C.c_int32 * (MAX_LAYERS + 1)), ('acts', C.c_int32 * MAX_LAYERS),
                ('w_off', C.c_int32 * MAX_LAYERS), ('b_off', C.c_int32 * MAX_LAYERS), ('row_stride', C.c_int32),
                ('n_actions', C.c_int32), ('n_features', C.c_int32)]


class ForwardArgs(C.Structure):
    _fields_ = [('net', NetDesc), ('params', C.c_void_p), ('policy_lo', C.c_int32), ('n_pol', C.c_int32),
                ('x', C.c_void_p), ('B', C.c_int32), ('psi_out', C.c_void_p), ('acts_out', C.c_void_p * MAX_LAYERS),
                ('sel_actions', C.c_void_p), ('sel_keys', C.c_void_p), ('sel_key_stride', C.c_int32),
                ('sel_out', C.c_void_p), ('w', C.c_void_p), ('n_w', C.c_int32), ('w_diag', C.c_int32),
                ('key_action', C.c_void_p), ('key_task', C.c_void_p), ('task_base', C.c_int32), ('q_out', C.c_void_p),
                ('mode', C.c_int32), ('acts_bf16_out', C.c_void_p), ('relu_mask_out', C.c_void_p)]


class TdArgs(C.Structure):
    _fields_ = [('variant', C.c_int32), ('n_pol', C.c_int32), ('B', C.c_int32), ('S', C.c_int32), ('A', C.c_int32),
                ('D', C.c_int32), ('G', C.c_int32), ('beta', C.c_float), ('cur_sel', C.c_void_p), ('next_sel', C.c_void_p),
                ('phis', C.c_void_p), ('rs', C.c_void_p), ('gammas', C.c_void_p), ('states', C.c_void_p),
                ('next_states', C.c_void_p), ('w', C.c_void_p), ('g', C.c_void_p), ('h', C.c_void_p),
                ('w_stride', C.c_int32), ('g_stride', C.c_int32), ('d_out', C.c_void_p), ('loss_part', C.c_void_p),
                ('aux_grad_part', C.c_void_p), ('aux_len', C.c_int32), ('next_psi', C.c_void_p), ('next_keys', C.c_void_p),
                ('next_key_stride', C.c_int32), ('tsf_part', C.c_void_p), ('peer_keys', C.c_void_p), ('defer_expand', C.c_int32),
                ('tsf_mc', C.c_void_p), ('n_flows', C.c_int32)]


class ForwardTcJob(C.Structure):
    _fields_ = [('args', ForwardArgs), ('params_bf16', C.c_void_p), ('n_policies_total', C.c_int32), ('wq', C.c_void_p),
                ('bq', C.c_void_p)]


class BackwardArgs(C.Structure):
    _fields_ = [('net', NetDesc), ('params', C.c_void_p), ('policy_lo', C.c_int32), ('n_pol', C.c_int32),
                ('x', C.c_void_p), ('B', C.c_int32), ('acts', C.c_void_p * MAX_LAYERS), ('actions', C.c_void_p),
                ('d_out', C.c_void_p), ('dz', C.c_void_p * MAX_LAYERS), ('grad_part', C.c_void_p), ('n_split', C.c_int32)]


class BackwardTcArgs(C.Structure):
    _fields_ = [('net', NetDesc), ('params_bf16', C.c_void_p), ('n_policies_total', C.c_int32), ('policy_lo', C.c_int32),
                ('n_pol', C.c_int32), ('x', C.c_void_p), ('B', C.c_int32), ('acts_bf16', C.c_void_p), ('relu_masks', C.c_void_p), ('actions', C.c_void_p),
                ('d_out', C.c_void_p), ('dz_bf16', C.c_void_p), ('dzo_bf16', C.c_void_p), ('xo_bf16', C.c_void_p),
                ('grad_part', C.c_void_p), ('n_split', C.c_int32), ('xo_ready', C.c_int32), ('expand_td', C.c_void_p)]


class BackwardStreamArgs(C.Structure):
    _fields_ = [('net', NetDesc), ('precision', C.c_int32), ('shadow_t', C.c_void_p), ('wout_t', C.c_void_p),
                ('n_policies_total', C.c_int32), ('policy_lo', C.c_int32), ('n_pol', C.c_int32), ('x', C.c_void_p), ('B', C.c_int32),
                ('acts', C.c_void_p), ('relu_masks', C.c_void_p), ('actions', C.c_void_p), ('d_out', C.c_void_p), ('dz', C.c_void_p),
                ('dzo', C.c_void_p), ('xo', C.c_void_p), ('grad_part', C.c_void_p), ('n_split', C.c_int32)]


class InputGradArgs(C.Structure):
    _fields_ = [('net', NetDesc), ('precision', C.c_int32), ('params', C.c_void_p), ('policy_lo', C.c_int32), ('n_pol', C.c_int32),
                ('B', C.c_int32), ('dz0', C.c_void_p), ('dz0_part_stride', C.c_int64), ('dx', C.c_void_p)]


class StepPrepArgs(C.Structure):
    _fields_ = [('net', NetDesc), ('pack_params', C.c_void_p * 2), ('pack_out', C.c_void_p * 2), ('pack_lo', C.c_int32 * 2),
                ('pack_n', C.c_int32 * 2), ('keys', C.c_void_p), ('n_keys', C.c_int64), ('fold_params', C.c_void_p),
                ('fold_lo', C.c_int32), ('fold_n', C.c_int32), ('w', C.c_void_p), ('n_w', C.c_int32), ('w_diag', C.c_int32),
                ('wq', C.c_void_p), ('bq', C.c_void_p), ('x', C.c_void_p), ('B', C.c_int32), ('xo_bf16', C.c_void_p),
                ('copy_src', C.c_void_p * 6), ('copy_dst', C.c_void_p * 6), ('copy_bytes', C.c_int64 * 6),
                ('tsf_g', C.c_void_p), ('tsf_h', C.c_void_p), ('tsf_mc', C.c_void_p), ('tsf_g_stride', C.c_int32), ('tsf_G', C.c_int32),
                ('tsf_lo', C.c_int32), ('tsf_n', C.c_int32)]


class ReplayArgs(C.Structure):
    _fields_ = [('ring', C.c_void_p), ('row_stride', C.c_int64), ('S', C.c_int32), ('D', C.c_int32), ('B', C.c_int32),
                ('picks', C.c_void_p), ('states', C.c_void_p), ('actions', C.c_void_p), ('rewards', C.c_void_p),
                ('phis', C.c_void_p), ('next_states', C.c_void_p), ('gammas', C.c_void_p)]


class Cmd(C.Structure):
    _fields_ = [('op', C.c_int32), ('p', C.c_void_p * 5), ('i', C.c_int64 * 4)]


OP = dict(H2D=1, D2H=2, D2D=3, KEYS_FILL=4, PACK_BF16=5, FOLD_GPI=6, FORWARD=7, FORWARD_TC_JOBS=8, TD=9, BACKWARD=10,
          BACKWARD_TC=11, ADAM=12, EVENT=13, PEER_KEYS=14, SHARD_PACK=15, PEER_UNPACK=16, STEP_PREP=17, PACK_F32=19,
          FOLD_GPI_F32=20, FORWARD_STREAM=21, BACKWARD_STREAM=22, KEYS_DECODE=23)
OP_LAUNCHES = {13: 0, 0: 0, 1: 0, 2: 0, 3: 0, 4: 1, 5: 1, 6: 1, 7: 1, 8: 1, 9: 1, 10: 2, 11: 3, 12: 2, 14: 1, 15: 1, 16: 1, 17: 1,
               19: 1, 20: 1, 21: 1, 22: 3, 23: 1}
MAX_PEERS = 16
PEER_CHANNELS = 4
IPC_HANDLE_BYTES = 64


class PeerCtx(C.Structure):
    _fields_ = [('world', C.c_int32), ('rank', C.c_int32), ('flags', C.c_void_p * MAX_PEERS)]


class PeerKeysArgs(C.Structure):
    _fields_ = [('ctx', PeerCtx), ('epoch', C.c_int64), ('keys_all', C.c_void_p * MAX_PEERS), ('row_lo', C.c_int32),
                ('n_rows', C.c_int32), ('B', C.c_int32), ('keys_out', C.c_void_p)]


class PeerUnpackArgs(C.Structure):
    _fields_ = [('ctx', PeerCtx), ('epoch', C.c_int64), ('x', C.c_void_p * MAX_PEERS), ('nw', C.c_int32), ('nh', C.c_int32),
                ('w_all', C.c_void_p), ('h', C.c_void_p), ('h_prev', C.c_void_p), ('pack_w', C.c_void_p)]


class AdamSegment(C.Structure):
    _fields_ = [('param', C.c_void_p), ('param_stride', C.c_int64), ('m', C.c_void_p), ('m_stride', C.c_int64),
                ('v', C.c_void_p), ('v_stride', C.c_int64), ('grad_part', C.c_void_p), ('grad_pol_stride', C.c_int64),
                ('grad_part_stride', C.c_int64), ('n_part', C.c_int32), ('len', C.c_int32), ('lr', C.c_float),
                ('weight_decay', C.c_float), ('clamp_min', C.c_float), ('clamp_max', C.c_float)]


class AdamArgs(C.Structure):
    _fields_ = [('n_seg', C.c_int32), ('n_pol', C.c_int32), ('seg', AdamSegment * MAX_SEGMENTS), ('step', C.c_void_p),
                ('beta1', C.c_double), ('beta2', C.c_double), ('eps', C.c_double), ('loss_part', C.c_void_p),
                ('n_loss_part', C.c_int32), ('l1_scale', C.c_float), ('l2_scale', C.c_float), ('beta_loss', C.c_float),
                ('losses', C.c_void_p), ('sequential_shared', C.c_int32), ('consts', C.c_void_p), ('consts_next', C.c_void_p),
                ('fresh', C.c_int32), ('losses_host', C.c_void_p)]


class TargetArgs(C.Structure):
    _fields_ = [('N', C.c_int32), ('A', C.c_int32), ('D', C.c_int32), ('G', C.c_int32), ('S', C.c_int32), ('psi', C.c_void_p),
                ('next_psi', C.c_void_p), ('g', C.c_void_p), ('g_stride', C.c_int32), ('h', C.c_void_p), ('s', C.c_void_p), ('s1', C.c_void_p),
                ('phi', C.c_void_p), ('r', C.c_float), ('gamma', C.c_float), ('a', C.c_int32), ('a1', C.c_int32), ('beta', C.c_float),
                ('l1_coef', C.c_float), ('lr_w', C.c_float), ('wd_w', C.c_float), ('lr_omega', C.c_float), ('wd_omega', C.c_float),
                ('lr_omega_decay', C.c_float), ('w', C.c_void_p), ('omegas', C.c_void_p), ('w_m', C.c_void_p), ('w_v', C.c_void_p),
                ('o_m', C.c_void_p), ('o_v', C.c_void_p), ('step', C.c_void_p), ('epoch', C.c_void_p), ('losses', C.c_void_p)]


class G4Args(C.Structure):
    _fields_ = [('B', C.c_int32), ('A', C.c_int32), ('D', C.c_int32), ('cur_sel', C.c_void_p), ('next_sel', C.c_void_p), ('phi', C.c_void_p),
                ('rs', C.c_void_p), ('gammas', C.c_void_p), ('w', C.c_void_p), ('bias', C.c_void_p), ('coef', C.c_void_p),
                ('d_psi', C.c_void_p), ('d_phi', C.c_void_p), ('grad_small', C.c_void_p), ('losses', C.c_void_p)]


# every symbol include/sfgpi.h declares: name -> (restype, argtypes)
SYMBOLS = {
    'sfgpi_mlp_forward': (C.c_int, [C.POINTER(ForwardArgs), C.c_void_p]),
    'sfgpi_keys_fill': (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    'sfgpi_keys_decode': (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    'sfgpi_gpi_from_psi': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'sfgpi_td_partials': (C.c_int, [C.c_int32]),
    'sfgpi_td_step': (C.c_int, [C.POINTER(TdArgs), C.c_void_p]),
    'sfgpi_mlp_backward': (C.c_int, [C.POINTER(BackwardArgs), C.c_void_p]),
    'sfgpi_adam_step': (C.c_int, [C.POINTER(AdamArgs), C.c_void_p]),
    'sfgpi_adam_refresh': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_double, C.c_double, C.c_void_p]),
    'sfgpi_bf16_rows_per_policy': (C.c_int, [C.POINTER(NetDesc)]),
    'sfgpi_pack_bf16': (C.c_int, [C.POINTER(NetDesc), C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    'sfgpi_gpi_fold_rows': (C.c_int, [C.POINTER(NetDesc), C.c_int32]),
    'sfgpi_fold_gpi': (C.c_int, [C.POINTER(NetDesc), C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    'sfgpi_mlp_forward_tc': (C.c_int, [C.POINTER(ForwardArgs), C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    'sfgpi_bwd_tc_out_pad': (C.c_int, [C.POINTER(NetDesc)]),
    'sfgpi_bwd_tc_splits': (C.c_int, [C.c_int32, C.c_int32]),
    'sfgpi_mlp_backward_tc': (C.c_int, [C.POINTER(BackwardTcArgs), C.c_void_p]),
    'sfgpi_mlp_forward_tc_jobs': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    'sfgpi_f32_out_pad': (C.c_int, [C.POINTER(NetDesc)]),
    'sfgpi_pack_f32': (C.c_int, [C.POINTER(NetDesc), C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    'sfgpi_fold_gpi_f32': (C.c_int, [C.POINTER(NetDesc), C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                     C.c_void_p, C.c_void_p, C.c_void_p]),
    'sfgpi_mlp_forward_stream': (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    'sfgpi_mlp_backward_stream': (C.c_int, [C.POINTER(BackwardStreamArgs), C.c_void_p]),
    'sfgpi_mlp_input_grad': (C.c_int, [C.POINTER(InputGradArgs), C.c_void_p]),
    'sfgpi_g4_head': (C.c_int, [C.POINTER(G4Args), C.c_void_p]),
    'sfgpi_target_q': (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'sfgpi_target_adapt': (C.c_int, [C.POINTER(TargetArgs), C.c_void_p]),
    'sfgpi_lms_update': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_void_p]),
    'sfgpi_replay_gather': (C.c_int, [C.POINTER(ReplayArgs), C.c_void_p]),
    'sfgpi_run': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    'sfgpi_shard_pack': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    'sfgpi_shard_unpack': (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'sfgpi_step_prep': (C.c_int, [C.POINTER(StepPrepArgs), C.c_void_p]),
    'sfgpi_step_prep_launches': (C.c_int, [C.c_void_p]),
    'sfgpi_phi_head_partials': (C.c_int, [C.c_int32]),
    'sfgpi_phi_head': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'sfgpi_peer_alloc': (C.c_int, [C.c_int64, C.POINTER(C.c_void_p), C.c_void_p]),
    'sfgpi_peer_open': (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    'sfgpi_peer_close': (C.c_int, [C.c_void_p]),
    'sfgpi_peer_free': (C.c_int, [C.c_void_p]),
    'sfgpi_peer_reduce_keys': (C.c_int, [C.POINTER(PeerKeysArgs), C.c_void_p]),
    'sfgpi_peer_unpack': (C.c_int, [C.POINTER(PeerUnpackArgs), C.c_void_p]),
    'sfgpi_set_option': (C.c_int, [C.c_char_p, C.c_int32]),
    'sfgpi_trace_dump': (None, []),
    'sfgpi_trace_enable': (None, [C.c_int32]),
    'sfgpi_trace_read': (C.c_int, [C.c_void_p, C.c_int32]),
    'sfgpi_last_error': (C.c_char_p, []),
    'sfgpi_version': (C.c_int, []),
}

_lib = None
launch_count = 0          # kernels launched through the C ABI (bench.py reports it as gpu_launches)
LAUNCHES_PER_CALL = {'sfgpi_pack_bf16': 1, 'sfgpi_fold_gpi': 1, 'sfgpi_mlp_forward_tc': 1, 'sfgpi_mlp_forward': 1, 'sfgpi_keys_fill': 1, 'sfgpi_keys_decode': 1, 'sfgpi_gpi_from_psi': 1,
                     'sfgpi_td_step': 2, 'sfgpi_mlp_backward': 2, 'sfgpi_mlp_backward_tc': 3, 'sfgpi_adam_step': 2,
                     'sfgpi_step_prep': 1, 'sfgpi_mlp_backward_stream': 3,
    'sfgpi_peer_alloc': 0, 'sfgpi_peer_open': 0, 'sfgpi_peer_close': 0, 'sfgpi_peer_free': 0}


def lib():
    """Loads (building first if needed) libsfgpi.so.  Raises if that is impossible -- there is no other code path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build()
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(handle, name)           # AttributeError if the .so does not export a declared symbol
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def call(name, *args):
    global launch_count
    rc = getattr(lib(), name)(*args)
    if rc != 0:
        raise RuntimeError(f'{name} failed (rc={rc}): {lib().sfgpi_last_error().decode()}')
    launch_count += LAUNCHES_PER_CALL.get(name, 1)


def run(cmds, n, stream, launches):
    """One foreign call for a whole command list (sfgpi_run); `launches` = kernels it launches, for the bench's count."""
    global launch_count
    rc = lib().sfgpi_run(C.byref(cmds), n, stream)
    if rc != 0:
        raise RuntimeError(f'sfgpi_run failed (rc={rc}): {lib().sfgpi_last_error().decode()}')
    launch_count += launches


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())
