"""ctypes binding of libcacto_b200.so (include/cacto_b200.h).

The shared library is the product: if it is missing, or was built without a symbol the header
declares, importing this module raises -- there is no CPU fallback on this path.
"""
import ctypes as C
import os

import numpy as np

from . import robots

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('CACTO_B200_LIB', os.path.join(_HERE, 'libcacto_b200.so'))   # override: instrumented builds

SYSTEM_CODE = dict(single_integrator=0, double_integrator=1, car=2, car_park=3, manipulator=4, ur5=5)
MAX_NS, MAX_NA, MAX_JOINTS = 13, 6, 6


class Chain(C.Structure):
    _fields_ = [('n', C.c_int32), ('jtype', C.c_int32 * MAX_JOINTS), ('axis', C.c_int32 * MAX_JOINTS),
                ('p', (C.c_double * 3) * MAX_JOINTS), ('R', (C.c_double * 9) * MAX_JOINTS), ('mass', C.c_double * MAX_JOINTS),
                ('com', (C.c_double * 3) * MAX_JOINTS), ('inertia', (C.c_double * 6) * MAX_JOINTS), ('ee_p', C.c_double * 3),
                ('gravity', C.c_double)]


class SysParams(C.Structure):
    _fields_ = [('system', C.c_int32), ('nx', C.c_int32), ('ns', C.c_int32), ('na', C.c_int32), ('normalize', C.c_int32),
                ('pad_', C.c_int32), ('dt', C.c_double), ('state_norm', C.c_double * (MAX_NS + 3)),
                ('u_max', C.c_double * (MAX_NA + 2)), ('scale', C.c_double), ('offset', C.c_double), ('alpha', C.c_double),
                ('alpha2', C.c_double), ('w_b', C.c_double), ('target', C.c_double * 3), ('obs', C.c_double * 18),
                ('L_delta', C.c_double), ('tau_delta', C.c_double), ('k_db', C.c_double), ('check_points', C.c_double * 20),
                ('w_running', C.c_double * 8), ('w_terminal', C.c_double * 8), ('chain', Chain)]


def make_sys_params(conf):
    """Pack the scalars of a conf (reference conf module or cacto_b200.conf namespace) that the
    kernels read into the POD ``cacto_sys_params``."""
    P = SysParams()
    sid = conf.system_id
    P.system = SYSTEM_CODE[sid]
    P.nx, P.ns, P.na = int(conf.nx), int(conf.nb_state), int(conf.nb_action)
    P.normalize = int(bool(conf.NORMALIZE_INPUTS))
    P.dt = float(conf.dt)
    for i, v in enumerate(np.asarray(conf.state_norm_arr, dtype=float)):
        P.state_norm[i] = v
    for i, v in enumerate(np.asarray(conf.u_max, dtype=float)):
        P.u_max[i] = v
    P.offset, P.scale = float(conf.cost_funct_param[0]), float(conf.cost_funct_param[1])     # environment.py:43-44
    P.alpha, P.alpha2 = float(conf.soft_max_param[0]), float(conf.soft_max_param[1])
    P.w_b = float(conf.w_b)
    for i, v in enumerate(np.asarray(conf.TARGET_STATE, dtype=float)):
        P.target[i] = v
    for i, v in enumerate(np.asarray(conf.obs_param, dtype=float)):
        P.obs[i] = v
    P.L_delta = float(getattr(conf, 'L_delta', 1.0))
    P.tau_delta = float(getattr(conf, 'tau_delta', 1.0))
    P.k_db = float(getattr(conf, 'k_db', 1.0))
    if hasattr(conf, 'check_points_BF'):
        for i, v in enumerate(np.asarray(conf.check_points_BF, dtype=float).reshape(-1)):
            P.check_points[i] = v
    for i, v in enumerate(np.asarray(conf.cost_weights_running, dtype=float)):
        P.w_running[i] = v
    for i, v in enumerate(np.asarray(conf.cost_weights_terminal, dtype=float)):
        P.w_terminal[i] = v
    P.chain.gravity = robots.GRAVITY
    if sid in robots.CHAINS:
        ch = robots.CHAINS[sid]
        P.chain.n = len(ch['joints'])
        for i, j in enumerate(ch['joints']):
            P.chain.jtype[i], P.chain.axis[i], P.chain.mass[i] = j['kind'], j['axis'], j['mass']
            for k in range(3):
                P.chain.p[i][k] = j['xyz'][k] + (ch['base'][k] if i == 0 else 0.0)
                P.chain.com[i][k] = j['com'][k]
            for k, v in enumerate(robots.rpy_matrix(*j['rpy'])):
                P.chain.R[i][k] = v
            for k in range(6):
                P.chain.inertia[i][k] = j['inertia'][k]
        for k in range(3):
            P.chain.ee_p[k] = ch['ee'][k]
    return P


_SIGNATURES = {
    'cacto_abi_version': (C.c_int32, []),
    'cacto_actor_param_count': (C.c_int64, [C.c_int32, C.c_int32]),
    'cacto_critic_param_count': (C.c_int64, [C.c_int32]),
    'cacto_dyn_step': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_dyn_derivative': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_dyn_augmented': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                      C.c_void_p]),
    'cacto_ee_position': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_reward': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                               C.c_int64, C.c_void_p]),
    'cacto_rollout': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
    C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_actor_tc_image_floats': (C.c_int64, []),
    'cacto_actor_tc_prepare': (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    'cacto_rollout_tc': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_actor_tc16_image_bytes': (C.c_int64, []),
    'cacto_actor_tc16_prepare': (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    'cacto_rollout_tc16': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_backward_pass_workspace_bytes': (C.c_int64, [C.c_int32, C.c_int32, C.c_int64]),
    'cacto_backward_pass': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_void_p, C.c_void_p,
                                      C.c_void_p]),
    'cacto_ddp_workspace_bytes': (C.c_int64, [C.c_int32, C.c_int32, C.c_int64, C.c_int32]),
    'cacto_ddp_init': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64] + [C.c_void_p] * 5),
    'cacto_ddp_iterate': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_double] +
                          [C.c_void_p] * 5),
    'cacto_copy2d_to_host':(C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p]),
    'cacto_copy3d_to_host': (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                       C.c_void_p]),
    'cacto_narrow_f64_to_f32': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_host_mt19937_random': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    'cacto_mlp_forward_generic': (C.c_int, [C.c_void_p] * 6 + [C.c_int64, C.c_void_p]),
    'cacto_critic_grad_generic': (C.c_int, [C.c_void_p] * 4 + [C.c_float, C.c_int] + [C.c_void_p] * 6 + [C.c_float] + [C.c_void_p] * 5 +
                                  [C.c_int64, C.c_void_p]),
    'cacto_actor_grad_generic': (C.c_int, [C.c_void_p] * 9 + [C.c_float, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_adam_step_peer': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_float, C.c_void_p, C.c_int32,
                                       C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_void_p]),
    'cacto_peer_alloc': (C.c_int, [C.c_int64, C.POINTER(C.c_void_p)]),
    'cacto_peer_free': (C.c_int, [C.c_void_p]),
    'cacto_peer_export': (C.c_int, [C.c_void_p, C.c_void_p]),
    'cacto_peer_open': (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    'cacto_peer_close': (C.c_int, [C.c_void_p]),
    'cacto_actor_width_param_count': (C.c_int64, [C.c_int32] * 4),
    'cacto_rollout_width': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_actor_forward_width': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_actor_grad_width': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32] + [C.c_void_p] * 4 + [C.c_float, C.c_void_p, C.c_void_p, C.c_int64,
                                                                                                        C.c_void_p]),
    'cacto_actor_forward': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_critic_forward': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_critic_grad': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int] + [C.c_void_p] * 6 +
    [C.c_float] + [C.c_void_p] * 5 + [C.c_int64, C.c_void_p]),
    'cacto_actor_grad': (C.c_int, [C.c_void_p] * 7 + [C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_update_tc_workspace_bytes': (C.c_int64, [C.c_int64, C.c_int32, C.c_int32]),
    'cacto_critic_grad_tc': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int] + [C.c_void_p] * 6 + [C.c_float] + [C.c_void_p] * 5 +
                             [C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_actor_grad_tc': (C.c_int, [C.c_void_p] * 5 + [C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_det_partials_floats': (C.c_int64, [C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    'cacto_critic_grad_det': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int] + [C.c_void_p] * 6 +
                              [C.c_float] + [C.c_void_p] * 5 + [C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_actor_grad_det': (C.c_int, [C.c_void_p] * 7 + [C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_actor_grad_width_det': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32] + [C.c_void_p] * 4 + [C.c_float, C.c_void_p, C.c_void_p,
                                                                                                            C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_critic_grad_tc_det': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int] + [C.c_void_p] * 6 + [C.c_float] +
                                 [C.c_void_p] * 5 + [C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    'cacto_actor_grad_tc_det': (C.c_int, [C.c_void_p] * 5 + [C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64,
                                          C.c_void_p]),
    'cacto_adam_schedule': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    'cacto_adam_schedule2': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_float, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    'cacto_adam_step': (C.c_int, [C.c_void_p] * 4 + [C.c_float, C.c_void_p] + [C.c_float] * 3 + [C.c_void_p, C.c_float, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                  C.c_int64, C.c_void_p]),
    'cacto_transpose_params': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    'cacto_segtree_update': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    'cacto_segtree_reduce': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    'cacto_segtree_sample': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]),
    'cacto_segtree_find': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    'cacto_host_pow': (C.c_int, [C.c_void_p, C.c_double, C.c_void_p, C.c_int64]),
    'cacto_buffer_gather': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32] + [C.c_void_p] * 8 + [C.c_void_p]),
    'cacto_peak_fma_fp32': (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    'cacto_rtg_window': (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32] +
                         [C.c_void_p] * 6 + [C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

MLP_MAX_LAYERS = 8
ACT_CODES = {'linear': 0, 'sin': 1, 'elu': 2, 'leaky': 3}


class MlpDesc(C.Structure):
    """cacto_mlp_desc of include/cacto_b200.h."""
    _fields_ = [('n_layers', C.c_int32), ('dims', C.c_int32 * (MLP_MAX_LAYERS + 1)), ('act', C.c_int32 * MLP_MAX_LAYERS)]


def make_mlp_desc(dims, acts):
    assert len(acts) == len(dims) - 1 <= MLP_MAX_LAYERS
    d = MlpDesc()
    d.n_layers = len(acts)
    for i, v in enumerate(dims):
        d.dims[i] = int(v)
    for i, a in enumerate(acts):
        d.act[i] = ACT_CODES[a]
    return d


def load_library(path=LIB_PATH):
    if not os.path.exists(path):
        raise ImportError(f'{path} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                          '(there is no CPU fallback for the CACTO hot path)')
    lib = C.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so lacks a declared symbol
        fn.restype, fn.argtypes = res, args
    if lib.cacto_abi_version() != 1:
        raise ImportError('libcacto_b200.so ABI version mismatch')
    return lib


lib = load_library()

_ERR = {-1: 'bad argument', -2: 'unknown system', -3: 'unsupported dtype', -4: 'bad size', -5: 'misaligned buffer'}


def check(rc, what=''):
    if rc == 0:
        return
    if rc < 0:
        raise RuntimeError(f'cacto_b200 {what}: {_ERR.get(rc, rc)}')
    raise RuntimeError(f'cacto_b200 {what}: CUDA error {rc}')


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)
