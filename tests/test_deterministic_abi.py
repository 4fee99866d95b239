"""Boundary of the deterministic gradient entry points (cacto_*_grad_det, include/cacto_b200.h): exported and declared symbols, the
partials-workspace size and its cap, argument checks that return negative codes before any launch, the element-count checks of
the torch shims, and the critic types that refuse the mode.  No GPU needed."""
import ctypes as C
import os
import re

import pytest
import torch

from cacto_b200 import _lib as L
from cacto_b200.conf import get_conf

NEW = ('cacto_det_partials_floats', 'cacto_critic_grad_det', 'cacto_actor_grad_det', 'cacto_actor_grad_width_det', 'cacto_critic_grad_tc_det',
       'cacto_actor_grad_tc_det')
E_ARG, E_SYSTEM, E_SIZE, E_ALIGN = -1, -2, -4, -5
CRITIC, ACTOR, ACTOR_WIDTH, CRITIC_TC, ACTOR_TC = 0, 1, 2, 3, 4
TC_SLICE = 648
MAX_SLICES = 296


def test_new_symbols_are_declared_and_exported():
    hdr = open(os.path.join(os.path.dirname(L.__file__), '..', 'include', 'cacto_b200.h')).read()
    for name in NEW:
        assert re.search(r'\b%s\(' % name, hdr), name
        assert name in L.EXPORTED_SYMBOLS
        assert getattr(L.lib, name) is not None
    assert re.search(r'#define CACTO_DET_MAX_SLICES %d\b' % MAX_SLICES, hdr)
    from cacto_b200.ops import OP_NAMES, ops
    for op in ('det_partials_floats', 'critic_grad_det', 'actor_grad_det', 'actor_grad_width_det', 'critic_grad_tc_det', 'actor_grad_tc_det'):
        assert op in OP_NAMES and hasattr(ops, op)
    assert L.lib.cacto_abi_version() == 1


def _stride(n):
    return (n + 1 + 3) // 4 * 4


def _tile(B):
    return 16 if B >= 16 * 148 else (2 if B <= 2 * 148 else (4 if B <= 4 * 148 else 8))


@pytest.mark.parametrize('B', [1, 64, 128, 297, 500, 2000, 4096, 16384, 10 ** 6])
def test_partials_size(B):
    lib = L.lib
    ns, na = 7, 2
    nc, nact = lib.cacto_critic_param_count(ns), lib.cacto_actor_param_count(ns, na)
    slices = min(-(-B // _tile(B)), MAX_SLICES)
    assert lib.cacto_det_partials_floats(CRITIC, B, ns, na, 0, 0) == slices * _stride(nc)
    assert lib.cacto_det_partials_floats(ACTOR, B, ns, na, 0, 0) == slices * _stride(nact)
    nw = lib.cacto_actor_width_param_count(ns, na, 128, 37)
    wt = 4 if B <= 4 * 148 else 16
    assert lib.cacto_det_partials_floats(ACTOR_WIDTH, B, ns, na, 128, 37) == min(-(-B // wt), MAX_SLICES) * _stride(nw)
    tc_slices = min(-(-B // 128), MAX_SLICES)         # one slice per CTA of the tcgen05 kernels' grid, 3 / 2 kernels with column sums
    assert lib.cacto_det_partials_floats(CRITIC_TC, B, ns, na, 0, 0) == 3 * tc_slices * TC_SLICE
    assert lib.cacto_det_partials_floats(ACTOR_TC, B, ns, na, 0, 0) == 2 * tc_slices * TC_SLICE


def test_partials_size_stays_flat_above_the_cap():
    lib = L.lib
    for net in (CRITIC, ACTOR, CRITIC_TC, ACTOR_TC):
        full = (128 if net >= CRITIC_TC else 16) * MAX_SLICES          # the batch from which every slice is in use
        cap = lib.cacto_det_partials_floats(net, full, 7, 2, 0, 0)
        assert lib.cacto_det_partials_floats(net, full - 128, 7, 2, 0, 0) < cap
        for B in (full + 1, 2 * full, 10 ** 6, 10 ** 8):
            assert lib.cacto_det_partials_floats(net, B, 7, 2, 0, 0) == cap
    # the manipulator at the reference batch size: 32 slices of the critic's 29 633 parameters (+ the loss partial, padded)
    assert lib.cacto_det_partials_floats(CRITIC, 64, 7, 2, 0, 0) == 32 * 29636
    assert lib.cacto_det_partials_floats(CRITIC, 16384, 7, 2, 0, 0) * 4 < 40 * 2 ** 20


def test_partials_size_rejects_bad_arguments():
    lib = L.lib
    assert lib.cacto_det_partials_floats(5, 64, 7, 2, 0, 0) == E_SIZE
    assert lib.cacto_det_partials_floats(CRITIC_TC, -1, 7, 2, 0, 0) == E_SIZE
    assert lib.cacto_det_partials_floats(CRITIC, -1, 7, 2, 0, 0) == E_SIZE
    assert lib.cacto_det_partials_floats(CRITIC, 64, 1, 2, 0, 0) == E_SIZE
    assert lib.cacto_det_partials_floats(ACTOR, 64, 7, 0, 0, 0) == E_SIZE
    for h1, h2 in ((0, 64), (513, 64), (64, 0), (64, 513)):
        assert lib.cacto_det_partials_floats(ACTOR_WIDTH, 64, 7, 2, h1, h2) == E_SIZE


def test_bad_arguments_are_rejected_without_launching():
    lib = L.lib
    conf = get_conf('manipulator')
    P = L.make_sys_params(conf)
    pp = C.byref(P)
    ns, na = conf.nb_state, conf.nb_action
    null = C.c_void_p(0)
    a = C.c_void_p(4096)           # never dereferenced: every call below is refused before a launch
    mis = C.c_void_p(4100)         # not 16-byte aligned
    B = 64
    nc = lib.cacto_det_partials_floats(CRITIC, B, ns, na, 0, 0)
    na_ = lib.cacto_det_partials_floats(ACTOR, B, ns, na, 0, 0)
    nw = lib.cacto_det_partials_floats(ACTOR_WIDTH, B, ns, na, 64, 64)

    def critic(part=a, n=nc, grad=a, p=pp, bsz=B):
        return lib.cacto_critic_grad_det(p, a, a, a, 1e-2, 0, a, a, a, a, a, a, 1.0, grad, a, a, a, null, bsz, part, n, null)

    def actor(part=a, n=na_, grad=a, p=pp, bsz=B):
        return lib.cacto_actor_grad_det(p, a, a, a, a, a, a, 1.0, grad, null, bsz, part, n, null)

    def width(part=a, n=nw, grad=a, p=pp, h1=64, bsz=B):
        return lib.cacto_actor_grad_width_det(p, a, h1, 64, a, a, a, a, 1.0, grad, null, bsz, part, n, null)

    for f in (critic, actor, width):
        assert f(p=null) == E_ARG
        assert f(part=null) == E_ARG
        assert f(grad=null) == E_ARG
        assert f(part=mis) == E_ALIGN
        assert f(grad=mis) == E_ALIGN
        assert f(bsz=-1) == E_SIZE
        assert f(bsz=0) == 0                 # an empty batch is a no-op
    assert critic(n=nc - 1) == E_SIZE
    assert actor(n=na_ - 1) == E_SIZE
    assert width(n=nw - 1) == E_SIZE
    assert width(h1=513) == E_SIZE
    # the critic's other inputs
    assert lib.cacto_critic_grad_det(pp, a, null, a, 1e-2, 0, a, a, a, a, a, a, 1.0, a, a, a, a, null, B, a, nc, null) == E_ARG
    assert lib.cacto_critic_grad_det(pp, a, a, a, 1e-2, 0, a, null, a, a, a, a, 1.0, a, a, a, a, null, B, a, nc, null) == E_ARG    # state_next, TD mode
    assert lib.cacto_critic_grad_det(pp, a, a, a, 1e-2, 0, a, a, a, null, a, a, 1.0, a, a, a, a, null, B, a, nc, null) == E_ARG    # dVdx with w_S != 0
    assert lib.cacto_critic_grad_det(pp, mis, a, a, 1e-2, 0, a, a, a, a, a, a, 1.0, a, a, a, a, null, B, a, nc, null) == E_ALIGN
    # the tcgen05 engine: the workspace checks of cacto_*_grad_tc first, then the partials
    ntc = lib.cacto_det_partials_floats(CRITIC_TC, B, ns, na, 0, 0)
    nta = lib.cacto_det_partials_floats(ACTOR_TC, B, ns, na, 0, 0)
    wsb = 1 << 40

    def critic_tc(part=a, n=ntc, ws=a, grad=a):
        return lib.cacto_critic_grad_tc_det(pp, a, a, 1e-2, 0, a, a, a, a, a, a, 1.0, grad, a, a, a, null, B, ws, wsb, part, n, null)

    def actor_tc(part=a, n=nta, ws=a, grad=a):
        return lib.cacto_actor_grad_tc_det(pp, a, a, a, a, 1.0, grad, null, B, ws, wsb, part, n, null)

    for f, n in ((critic_tc, ntc), (actor_tc, nta)):
        assert f(part=null) == E_ARG
        assert f(ws=null) == E_ARG
        assert f(grad=null) == E_ARG
        assert f(part=mis) == E_ALIGN
        assert f(grad=mis) == E_ALIGN
        assert f(n=n - 1) == E_SIZE
    assert lib.cacto_critic_grad_tc_det(pp, a, a, 1e-2, 0, a, a, a, a, a, a, 1.0, a, a, a, a, null, 0, a, wsb, a, 0, null) == 0
    P.system = 9
    assert actor() == E_SYSTEM
    assert width() == E_SYSTEM


def test_shims_reject_undersized_partials():
    from cacto_b200.ops import ops, sys_tensor
    conf = get_conf('manipulator')
    p = sys_tensor(L.make_sys_params(conf))
    ns, na, B = conf.nb_state, conf.nb_action, 5
    f32, f64 = torch.float32, torch.float64
    nc, nact = L.lib.cacto_critic_param_count(ns), L.lib.cacto_actor_param_count(ns, na)
    c, a, s, term = torch.zeros(nc, dtype=f32), torch.zeros(nact, dtype=f32), torch.zeros(B, ns, dtype=f32), torch.zeros(B, dtype=f64)
    v = torch.zeros(B, 1, dtype=f32)
    short = lambda net, h1=0, h2=0: torch.zeros(int(ops.det_partials_floats(net, B, ns, na, h1, h2)) - 1, dtype=f32)
    with pytest.raises(RuntimeError, match='partials'):
        ops.critic_grad_det(p, c, c, c, 1e-2, 0, s, s, v, s, v, v, 0.2, torch.zeros(nc, dtype=f32), v, v, v, None, short(CRITIC))
    with pytest.raises(RuntimeError, match='partials'):
        ops.actor_grad_det(p, a, a, c, c, s, term, 0.2, torch.zeros(nact, dtype=f32), None, short(ACTOR))
    nw = L.lib.cacto_actor_width_param_count(ns, na, 64, 37)
    w = torch.zeros(nw, dtype=f32)
    with pytest.raises(RuntimeError, match='partials'):
        ops.actor_grad_width_det(p, w, 64, 37, c, c, s, term, 0.2, torch.zeros(nw, dtype=f32), None, short(ACTOR_WIDTH, 64, 37))
    with pytest.raises(RuntimeError, match='grad'):
        ops.actor_grad_det(p, a, a, c, c, s, term, 0.2, torch.zeros(nact - 1, dtype=f32), None, torch.zeros(10 ** 6, dtype=f32))


class _Env:
    _p = _pt = None


@pytest.mark.parametrize('critic_type', ['elu', 'sine-elu', 'relu'])
def test_generic_critics_refuse_the_deterministic_mode(critic_type):
    from cacto_b200.NeuralNetwork import NN
    conf = get_conf('manipulator', critic_type=critic_type)
    with pytest.raises(ValueError, match='deterministic'):
        NN(_Env(), conf, 1e-2, seed=0, deterministic=True)


def test_deterministic_mode_keeps_the_engine_choice():
    from cacto_b200.NeuralNetwork import NN
    for det in (False, True):
        nn = NN.__new__(NN)
        nn.deterministic = det
        assert not nn._use_tc(64) and not nn._use_tc(2399) and nn._use_tc(2400) and nn._use_tc(16384)
        nn.update_engine = 'tc'
        assert nn._use_tc(64)
        nn.update_engine = 'fma'
        assert not nn._use_tc(16384)
