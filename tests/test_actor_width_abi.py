"""Boundary of the width-generic actor kernels (csrc/actor_width.cu): exported and declared symbols, argument checks that return
negative codes before any launch, and the element-count checks of the torch shims.  No GPU needed."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from cacto_b200 import _lib as L
from cacto_b200.conf import get_conf

NEW = ('cacto_actor_width_param_count', 'cacto_rollout_width', 'cacto_actor_forward_width', 'cacto_actor_grad_width')
E_ARG, E_SYSTEM, E_SIZE, E_ALIGN = -1, -2, -4, -5


def test_new_symbols_are_declared_and_exported():
    hdr = open(os.path.join(os.path.dirname(L.__file__), '..', 'include', 'cacto_b200.h')).read()
    for name in NEW:
        assert re.search(r'\b%s\(' % name, hdr), name
        assert name in L.EXPORTED_SYMBOLS
        assert getattr(L.lib, name) is not None
    from cacto_b200.ops import OP_NAMES, ops
    for op in ('rollout_width', 'actor_forward_width', 'actor_grad_width'):
        assert op in OP_NAMES and hasattr(ops, op)
    assert L.lib.cacto_abi_version() == 1


def test_param_count():
    lib = L.lib
    for ns, na in ((2, 1), (7, 2), (13, 6)):
        for h1, h2 in ((1, 1), (37, 100), (256, 256), (512, 512)):
            assert lib.cacto_actor_width_param_count(ns, na, h1, h2) == ns * h1 + h1 + h1 * h2 + h2 + h2 * na + na
        assert lib.cacto_actor_width_param_count(ns, na, 256, 256) == lib.cacto_actor_param_count(ns, na)
    for h1, h2 in ((0, 64), (64, 0), (513, 64), (64, 513), (-1, 4)):
        assert lib.cacto_actor_width_param_count(7, 2, h1, h2) == E_SIZE


def _params(system='manipulator'):
    P = L.make_sys_params(get_conf(system))
    return P, C.byref(P)


def test_bad_arguments_are_rejected_without_launching():
    lib = L.lib
    P, pp = _params()
    null = C.c_void_p(0)
    a = C.c_void_p(4096)           # never dereferenced: every call below is refused before a launch
    mis = C.c_void_p(4100)         # not 16-byte aligned
    for h1, h2 in ((0, 64), (513, 64), (64, 0), (64, 513)):
        assert lib.cacto_rollout_width(pp, a, h1, h2, a, a, 10, a, a, a, null, 4, null) == E_SIZE
        assert lib.cacto_actor_forward_width(pp, a, h1, h2, a, a, 4, null) == E_SIZE
        assert lib.cacto_actor_grad_width(pp, a, h1, h2, a, a, a, a, 1.0, a, null, 4, null) == E_SIZE
    # null pointers
    assert lib.cacto_rollout_width(null, a, 64, 64, a, a, 10, a, a, a, null, 4, null) == E_ARG
    assert lib.cacto_rollout_width(pp, null, 64, 64, a, a, 10, a, a, a, null, 4, null) == E_ARG
    assert lib.cacto_rollout_width(pp, a, 64, 64, null, a, 10, a, a, a, null, 4, null) == E_ARG
    assert lib.cacto_rollout_width(pp, a, 64, 64, a, a, 10, a, null, a, null, 4, null) == E_ARG   # controls with T_max > 0
    assert lib.cacto_actor_forward_width(pp, null, 64, 64, a, a, 4, null) == E_ARG
    assert lib.cacto_actor_forward_width(pp, a, 64, 64, a, null, 4, null) == E_ARG
    assert lib.cacto_actor_grad_width(pp, a, 64, 64, null, a, a, a, 1.0, a, null, 4, null) == E_ARG
    assert lib.cacto_actor_grad_width(pp, a, 64, 64, a, null, a, a, 1.0, a, null, 4, null) == E_ARG
    assert lib.cacto_actor_grad_width(pp, a, 64, 64, a, a, a, null, 1.0, a, null, 4, null) == E_ARG
    assert lib.cacto_actor_grad_width(pp, a, 64, 64, a, a, a, a, 1.0, null, null, 4, null) == E_ARG
    # misalignment
    assert lib.cacto_rollout_width(pp, mis, 64, 64, a, a, 10, a, a, a, null, 4, null) == E_ALIGN
    assert lib.cacto_actor_forward_width(pp, mis, 64, 64, a, a, 4, null) == E_ALIGN
    assert lib.cacto_actor_grad_width(pp, a, 64, 64, a, a, a, a, 1.0, mis, null, 4, null) == E_ALIGN
    assert lib.cacto_actor_grad_width(pp, a, 64, 64, a, mis, a, a, 1.0, a, null, 4, null) == E_ALIGN
    # sizes
    assert lib.cacto_rollout_width(pp, a, 64, 64, a, a, -1, a, a, a, null, 4, null) == E_SIZE
    assert lib.cacto_rollout_width(pp, a, 64, 64, a, a, 10, a, a, a, null, -1, null) == E_SIZE
    assert lib.cacto_actor_forward_width(pp, a, 64, 64, a, a, -1, null) == E_SIZE
    assert lib.cacto_actor_grad_width(pp, a, 64, 64, a, a, a, a, 1.0, a, null, -1, null) == E_SIZE
    # empty batches are no-ops; an unknown system is refused
    assert lib.cacto_rollout_width(pp, a, 64, 64, a, a, 10, a, a, a, null, 0, null) == 0
    assert lib.cacto_actor_grad_width(pp, a, 64, 64, a, a, a, a, 1.0, a, null, 0, null) == 0
    P.system = 9
    assert lib.cacto_rollout_width(pp, a, 64, 64, a, a, 10, a, a, a, null, 4, null) == E_SYSTEM
    assert lib.cacto_actor_grad_width(pp, a, 64, 64, a, a, a, a, 1.0, a, null, 4, null) == E_SYSTEM


def test_shims_reject_undersized_tensors():
    from cacto_b200.ops import ops, sys_tensor
    conf = get_conf('manipulator')
    p = sys_tensor(L.make_sys_params(conf))
    ns, na, B, T = conf.nb_state, conf.nb_action, 5, 4
    n = L.lib.cacto_actor_width_param_count(ns, na, 64, 37)
    f32, f64, i32 = torch.float32, torch.float64, torch.int32
    ics, hz = torch.zeros(B, ns, dtype=f64), torch.zeros(B, dtype=i32)
    st, ct, fl = torch.zeros((T + 1) * ns * B, dtype=f64), torch.zeros(T * na * B, dtype=f64), torch.zeros(B, dtype=i32)
    with pytest.raises(RuntimeError, match='actor'):
        ops.rollout_width(p, torch.zeros(n - 1, dtype=f32), 64, 37, ics, hz, T, st, ct, fl, None)
    with pytest.raises(RuntimeError, match='states'):
        ops.rollout_width(p, torch.zeros(n, dtype=f32), 64, 37, ics, hz, T, st[:-1], ct, fl, None)
    with pytest.raises(RuntimeError, match='controls'):
        ops.rollout_width(p, torch.zeros(n, dtype=f32), 64, 37, ics, hz, T, st, ct[:-1], fl, None)
    with pytest.raises(RuntimeError, match='outside'):
        ops.rollout_width(p, torch.zeros(n, dtype=f32), 513, 37, ics, hz, T, st, ct, fl, None)
    s = torch.zeros(B, ns, dtype=f32)
    with pytest.raises(RuntimeError, match='out'):
        ops.actor_forward_width(p, torch.zeros(n, dtype=f32), 64, 37, s, torch.zeros(B * na - 1, dtype=f32))
    nc = L.lib.cacto_critic_param_count(ns)
    c = torch.zeros(nc, dtype=f32)
    term = torch.zeros(B, dtype=f64)
    with pytest.raises(RuntimeError, match='grad'):
        ops.actor_grad_width(p, torch.zeros(n, dtype=f32), 64, 37, c, c, s, term, 0.2, torch.zeros(n - 1, dtype=f32), None)
    with pytest.raises(RuntimeError, match='critic_T'):
        ops.actor_grad_width(p, torch.zeros(n, dtype=f32), 64, 37, c, c[:-1], s, term, 0.2, torch.zeros(n, dtype=f32), None)
    with pytest.raises(RuntimeError, match='term'):
        ops.actor_grad_width(p, torch.zeros(n, dtype=f32), 64, 37, c, c, s, term[:-1], 0.2, torch.zeros(n, dtype=f32), None)
