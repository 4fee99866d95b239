"""PyTorch custom ops of the CACTO hot path: ``torch.ops.cacto.*`` (csrc/torch_ops.cpp, TORCH_LIBRARY(cacto, ...)).

Each op is a thin shim over the extern "C" symbol of the same name in libcacto_b200.so (include/cacto_b200.h): tensors in, raw
pointers + the current CUDA stream across the C boundary, a non-zero return code raised as RuntimeError.  The Python mirror of
the reference's modules (environment / NeuralNetwork / RL / replay_buffer / segment_tree / optim / rtg) calls the hot path through
these ops; what has no op yet (CUDA-IPC peer regions, the generic critic variants, the 3xTF32 rollout engine 'tf32', the TO
backward pass) goes through the same C ABI with ctypes (cacto_b200/_lib.py).

The shim library is part of the product: importing this module without it raises -- there is no fallback.
"""
import os

import torch

from . import _lib

_HERE = os.path.dirname(os.path.abspath(__file__))
OPS_PATH = os.environ.get('CACTO_B200_TORCH_LIB', os.path.join(_HERE, 'libcacto_b200_torch.so'))

if not os.path.exists(OPS_PATH):
    raise ImportError(f'{OPS_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                      '(the custom-op layer is the boundary of the CACTO hot path; there is no fallback)')
_lib.lib                                  # libcacto_b200.so is already loaded (the shim links against it)
torch.ops.load_library(OPS_PATH)
ops = torch.ops.cacto
if int(ops.abi_version()) != 1:
    raise ImportError('libcacto_b200_torch.so / libcacto_b200.so ABI version mismatch')

OP_NAMES = ('abi_version', 'dyn_step', 'dyn_derivative', 'dyn_augmented', 'ee_position', 'reward', 'rollout', 'actor_tc16_prepare', 'rollout_tc16',
            'rollout_width', 'actor_forward_width', 'actor_grad_width', 'actor_forward', 'critic_forward', 'critic_grad', 'actor_grad', 'update_tc_workspace_bytes', 'critic_grad_tc', 'actor_grad_tc',
            'det_partials_floats', 'critic_grad_det', 'actor_grad_det', 'actor_grad_width_det', 'critic_grad_tc_det', 'actor_grad_tc_det',
            'adam_schedule', 'adam_schedule2', 'adam_step', 'transpose_params', 'segtree_update', 'segtree_sample', 'buffer_gather', 'rtg_window')


def sys_tensor(params):
    """The POD ``cacto_sys_params`` (a ctypes structure, _lib.make_sys_params) as the CPU uint8 tensor the ops take."""
    return torch.frombuffer(bytearray(bytes(params)), dtype=torch.uint8).clone()
