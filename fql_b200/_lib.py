"""ctypes binding of libfql_b200.so (the C ABI declared in include/fql_b200.h).

There is deliberately NO fallback: if the shared library is missing or a call fails, this raises.  torch is used
by the callers only as the owner of device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libfql_b200.so')

NUM_INFO = 13
NUM_RAW = 16
NET_NAMES = ('actor_bc_flow', 'actor_onestep_flow', 'critic', 'target_critic')
NET_ACTOR_BC_FLOW, NET_ACTOR_ONESTEP_FLOW, NET_CRITIC, NET_TARGET_CRITIC = 0, 1, 2, 3
LEAF_KINDS = ('kernel', 'bias', 'scale', 'bias', 'kernel', 'bias', 'kernel', 'bias')
PRECISION_FP32, PRECISION_BF16_TC, PRECISION_BF16_ENC = 0, 1, 2


class FqlDims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        'batch', 'global_batch', 'obs_dim', 'action_dim', 'hidden', 'num_hidden', 'critic_layer_norm', 'actor_layer_norm',
        'q_agg_min', 'normalize_q_loss', 'flow_steps', 'num_seeds', 'precision')] + [('reserved', C.c_int32 * 3)]


class FqlHparams(C.Structure):
    _fields_ = [(n, C.c_float) for n in ('lr', 'beta1', 'beta2', 'eps', 'discount', 'tau', 'alpha', 'one_minus_beta1',
                                         'one_minus_beta2', 'one_minus_tau')] + [('reserved', C.c_float * 2)]


class FqlLeaf(C.Structure):
    _fields_ = [('net', C.c_int32), ('layer', C.c_int32), ('kind', C.c_int32), ('ens', C.c_int32), ('rows', C.c_int32),
                ('cols', C.c_int32), ('offset', C.c_int64)]


class FqlBatch(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('observations', 'actions', 'next_observations', 'rewards', 'masks', 'z_next', 'x0',
                                          't', 'z', 'z_metric')]


class FqlState(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('params', 'mu', 'nu', 'grads', 'count', 'shadow')]


DP_MAX_RANKS = 8


class FqlDpComm(C.Structure):
    _fields_ = [('rank', C.c_int32), ('world', C.c_int32), ('base', C.c_void_p * DP_MAX_RANKS), ('base_mc', C.c_void_p)]


class FqlTestOperand(C.Structure):
    _fields_ = [('ptr', C.c_void_p), ('inner', C.c_int32), ('rows', C.c_int32), ('ld', C.c_int64), ('g0', C.c_int32), ('s0', C.c_int64),
                ('g1', C.c_int32), ('s1', C.c_int64)]


class FqlTestPtr(C.Structure):
    _fields_ = [('base', C.c_void_p), ('s0', C.c_int64), ('s1', C.c_int64), ('ld', C.c_int32)]


TEST_GEMM_PTRS = ('bias', 'out_f', 'out_h', 'out_z', 'zin', 'act', 'xb', 'target', 'ln_s', 'ln_b', 'dbias', 'wmaster', 'dln_s', 'dln_b')


class FqlTestGemm(C.Structure):
    _fields_ = ([(n, C.c_int32) for n in ('mode', 'M', 'N', 'K', 'G0', 'G1', 'a_mn', 'b_mn', 'ksplit')] +
                [('A', FqlTestOperand), ('B', FqlTestOperand)] + [(n, FqlTestPtr) for n in TEST_GEMM_PTRS] +
                [(n, C.c_int32) for n in ('F', 'Adim', 'step', 'n_steps', 'clip')])


TC_MODE_STORE_F32, TC_MODE_FWD_HIDDEN, TC_MODE_DGRAD_GELU, TC_MODE_EULER, TC_MODE_WGRAD_LN = 0, 1, 2, 3, 4


class FqlError(RuntimeError):
    pass


_lib = None

_SIGS = {
    'fql_version': (C.c_int, []),
    'fql_last_error': (C.c_char_p, []),
    'fql_info_name': (C.c_char_p, [C.c_int]),
    'fql_context_create': (C.c_int, [C.POINTER(C.c_void_p)]),
    'fql_context_destroy': (C.c_int, [C.c_void_p]),
    'fql_launch_count': (C.c_longlong, [C.c_void_p]),
    'fql_arena_floats': (C.c_int64, [C.POINTER(FqlDims)]),
    'fql_layout': (C.c_int, [C.POINTER(FqlDims), C.POINTER(FqlLeaf), C.c_int32, C.POINTER(C.c_int32)]),
    'fql_workspace_bytes': (C.c_size_t, [C.POINTER(FqlDims)]),
    'fql_shadow_bytes': (C.c_size_t, [C.POINTER(FqlDims)]),
    'fql_forward_workspace_bytes': (C.c_size_t, [C.POINTER(FqlDims), C.c_int32]),
    'fql_update_step': (C.c_int, [C.c_void_p, C.POINTER(FqlDims), C.POINTER(FqlHparams), C.POINTER(FqlBatch), C.POINTER(FqlState),
                                  C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    'fql_step_grads': (C.c_int, [C.c_void_p, C.POINTER(FqlDims), C.POINTER(FqlHparams), C.POINTER(FqlBatch), C.POINTER(FqlState),
                                 C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    'fql_step_apply': (C.c_int, [C.c_void_p, C.POINTER(FqlDims), C.POINTER(FqlHparams), C.POINTER(FqlState), C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    'fql_step_apply_gathered': (C.c_int, [C.c_void_p, C.POINTER(FqlDims), C.POINTER(FqlHparams), C.POINTER(FqlState), C.c_void_p, C.c_int32,
                                          C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    'fql_dp_symmetric_bytes': (C.c_size_t, [C.POINTER(FqlDims), C.c_int32]),
    'fql_dp_attach': (C.c_int, [C.c_void_p, C.POINTER(FqlDims), C.POINTER(FqlDpComm)]),
    'fql_dp_allreduce': (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_void_p]),
    'fql_conv3x3_workspace_bytes': (C.c_size_t, []),
    'fql_conv3x3_bf16': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    'fql_conv3x3_wgrad_bf16': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    'fql_test_tc_gemm': (C.c_int, [C.POINTER(FqlTestGemm), C.c_void_p]),
    'fql_test_act_ln_bf16': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    'fql_test_ln_bwd_bf16': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32,
                                       C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_void_p]),
    'fql_test_gelu_bwd_bf16': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                         C.c_int64, C.c_int64, C.c_void_p]),
    'fql_test_colsum_bf16': (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_int64,
                                       C.c_void_p]),
    'fql_set_early_grads_event':(C.c_int, [C.c_void_p, C.c_void_p]),
    'fql_early_grads_floats': (C.c_int64, [C.POINTER(FqlDims)]),
    'fql_total_loss': (C.c_int, [C.c_void_p, C.POINTER(FqlDims), C.POINTER(FqlHparams), C.POINTER(FqlBatch), C.POINTER(FqlState),
                                 C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    'fql_sample_actions': (C.c_int, [C.c_void_p, C.POINTER(FqlDims), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    'fql_compute_flow_actions': (C.c_int, [C.c_void_p, C.POINTER(FqlDims), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    'fql_mlp_forward': (C.c_int, [C.c_void_p, C.POINTER(FqlDims), C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                  C.c_void_p, C.c_size_t, C.c_void_p]),
    'fql_target_update': (C.c_int, [C.POINTER(FqlDims), C.POINTER(FqlHparams), C.c_void_p, C.c_void_p, C.c_void_p]),
    'fql_debug_stamps': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    'fql_refresh_shadow': (C.c_int, [C.POINTER(FqlDims), C.c_void_p, C.c_void_p, C.c_void_p]),
    'fql_gather_rows': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    'fql_gather_frames': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                    C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    'fql_fill_noise': (C.c_int, [C.POINTER(FqlDims), C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    'fql_fill_noise_rows': (C.c_int, [C.POINTER(FqlDims), C.c_uint64, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
}
EXPORTS = tuple(_SIGS)


def lib():
    """Load (once) and return the shared library.  Raises if it has not been built: there is no CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FqlError(f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                           f'or `make -C fql_b200/csrc`. fql_b200 has no CPU or PyTorch fallback.')
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def check(rc, what=''):
    if rc != 0:
        raise FqlError(f'{what}: {lib().fql_last_error().decode()}')


def make_dims(batch, obs_dim, action_dim, *, global_batch=None, hidden=512, num_hidden=4, critic_layer_norm=True,
              actor_layer_norm=False, q_agg='mean', normalize_q_loss=False, flow_steps=10, num_seeds=1, precision=PRECISION_FP32,
              image=None):
    d = FqlDims()
    d.batch, d.global_batch = int(batch), int(global_batch if global_batch is not None else batch)
    d.obs_dim, d.action_dim, d.hidden, d.num_hidden = int(obs_dim), int(action_dim), int(hidden), int(num_hidden)
    d.critic_layer_norm, d.actor_layer_norm = int(bool(critic_layer_norm)), int(bool(actor_layer_norm))
    d.q_agg_min, d.normalize_q_loss = int(q_agg == 'min'), int(bool(normalize_q_loss))
    d.flow_steps, d.num_seeds, d.precision = int(flow_steps), int(num_seeds), int(precision)
    if image is not None:  # (H, W, C) uint8 observations through impala_small; obs_dim is then the encoder width 512
        d.reserved[0], d.reserved[1], d.reserved[2] = int(image[0]), int(image[1]), int(image[2])
    return d


def make_hparams(lr=3e-4, discount=0.99, tau=0.005, alpha=300.0, beta1=0.9, beta2=0.999, eps=1e-8):
    h = FqlHparams()
    h.lr, h.beta1, h.beta2, h.eps, h.discount, h.tau, h.alpha = lr, beta1, beta2, eps, discount, tau, alpha
    h.one_minus_beta1, h.one_minus_beta2, h.one_minus_tau = 1.0 - beta1, 1.0 - beta2, 1.0 - tau  # double, then rounded
    return h


def layout(dims):
    """[(net_name, layer, kind_name, ens, rows, cols, offset)] in arena order + floats per seed."""
    l = lib()
    n = C.c_int32(0)
    check(l.fql_layout(C.byref(dims), None, 0, C.byref(n)), 'fql_layout')
    arr = (FqlLeaf * n.value)()
    check(l.fql_layout(C.byref(dims), arr, n.value, C.byref(n)), 'fql_layout')
    out = []
    for lf in arr:
        if lf.kind < 4:
            path = (('LayerNorm' if lf.kind >= 2 else 'Dense') + f'_{lf.layer}',)
        elif lf.kind < 6:     # encoder convolution: stack_blocks_<i>/Conv_<j>  (utils/encoders.py:17-57)
            path = ('encoder', f'stack_blocks_{lf.layer // 3}', f'Conv_{lf.layer % 3}')
        else:                 # encoder head: MLP_0/Dense_0 (utils/encoders.py:98)
            path = ('encoder', 'MLP_0', 'Dense_0')
        shape = None
        if lf.kind == 4:      # HWIO [3,3,cin,cout]
            shape = (3, 3, lf.rows // 9, lf.cols)
        out.append(dict(net=NET_NAMES[lf.net], module=path[-1], path=path, name=LEAF_KINDS[lf.kind], ens=lf.ens, rows=lf.rows, cols=lf.cols,
                        offset=lf.offset, is_kernel=lf.kind in (0, 4, 6), shape=shape, kind=lf.kind))
    return out, int(l.fql_arena_floats(C.byref(dims)))
