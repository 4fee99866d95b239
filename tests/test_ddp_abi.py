"""Boundary of the iLQR TO solver (csrc/ddp.cu): exported and declared symbols, workspace sizes, the header's constants against the
oracle's, and argument checks that return negative codes before any launch.  No GPU needed."""
import ctypes as C
import os
import re

import pytest

from cacto_b200 import _lib as L
from cacto_b200.conf import SYSTEM_IDS, get_conf
from oracle import ddp as oddp

NEW = ('cacto_ddp_workspace_bytes', 'cacto_ddp_init', 'cacto_ddp_iterate')
E_ARG, E_SYSTEM, E_SIZE, E_ALIGN = -1, -2, -4, -5
HDR = open(os.path.join(os.path.dirname(L.__file__), '..', 'include', 'cacto_b200.h')).read()


def test_new_symbols_are_declared_and_exported():
    for name in NEW:
        assert re.search(r'\b%s\(' % name, HDR), name
        assert name in L.EXPORTED_SYMBOLS
        assert getattr(L.lib, name) is not None
    assert L.lib.cacto_abi_version() == 1


def test_header_constants_match_the_oracle_and_the_host():
    from cacto_b200.TO import TO_DDP
    define = lambda n: float(re.search(r'#define CACTO_DDP_%s (\S+)' % n, HDR).group(1))
    assert define('N_ALPHA') == oddp.N_ALPHA == TO_DDP.N_ALPHA
    assert define('HISTORY') == oddp.HISTORY == TO_DDP.HISTORY
    assert define('TRAJ_DOUBLES') == TO_DDP.TRAJ_DOUBLES
    for n in ('C1', 'MU_INIT', 'MU_MIN', 'MU_MAX', 'MU_FACTOR'):
        assert define(n) == getattr(oddp, n), n
    for n, v in (('RUNNING', 0), ('CONVERGED', 1), ('FAILED', 2)):
        assert re.search(r'CACTO_DDP_%s = %d\b' % (n, v), HDR) and getattr(oddp, n) == v == getattr(TO_DDP, n)
    for n in ('BACKWARD_FAILED', 'NO_STEP', 'CONVERGED', 'NOT_RUN'):
        assert int(re.search(r'CACTO_DDP_H_%s = (-\d+)' % n, HDR).group(1)) == getattr(oddp, 'H_' + n)


@pytest.mark.parametrize('system', SYSTEM_IDS)
def test_workspace_bytes(system):
    conf = get_conf(system)
    nx, na = conf.nb_state - 1, conf.nb_action
    knot = nx + 2 * nx * nx + nx * na + 2 * na + na + na * nx               # K6's block, then k and K
    for K, E in ((0, 0), (1, 1), (21, 3), (10 ** 6, 4096)):
        assert L.lib.cacto_ddp_workspace_bytes(nx, na, K, E) == 8 * (knot * K + 24 * E)
    assert L.lib.cacto_ddp_workspace_bytes(nx, na, 5, 1) - L.lib.cacto_backward_pass_workspace_bytes(nx, na, 5) == 8 * (5 * (na + na * nx) + 24)
    for args in ((0, na, 4, 1), (nx, 0, 4, 1), (nx, na, -1, 1), (nx, na, 4, -1)):
        assert L.lib.cacto_ddp_workspace_bytes(*args) == E_SIZE


def test_bad_arguments_are_rejected_without_launching():
    lib = L.lib
    P = L.make_sys_params(get_conf('car'))
    pp = C.byref(P)
    null = C.c_void_p(0)
    a = C.c_void_p(4096)           # never dereferenced: every call below is refused (or a no-op) before a launch
    mis = C.c_void_p(4100)
    init = lambda p=pp, off=a, E=3, s=a, u=a, K=12, ws=a, c=a, st=a, it=a: lib.cacto_ddp_init(p, off, E, s, u, K, ws, c, st, it, null)
    iterate = lambda p=pp, off=a, E=3, s=a, u=a, K=12, n=4, ws=a, c=a, st=a, it=a: lib.cacto_ddp_iterate(p, off, E, s, u, K, n, 1e-8, ws, c, st, it, null)
    # null pointers
    assert init(p=null) == E_ARG and iterate(p=null) == E_ARG
    for kw in ('off', 's', 'u', 'ws', 'c', 'st', 'it'):
        assert init(**{kw: null}) == E_ARG, kw
        assert iterate(**{kw: null}) == E_ARG, kw
    # sizes
    assert init(E=-1) == E_SIZE and iterate(E=-1) == E_SIZE
    assert init(K=-1) == E_SIZE and iterate(K=-1) == E_SIZE
    assert iterate(n=-1) == E_SIZE
    # alignment of the workspace
    assert init(ws=mis) == E_ALIGN and iterate(ws=mis) == E_ALIGN
    # empty work is a no-op
    assert init(E=0) == 0 and iterate(E=0) == 0 and iterate(n=0) == 0 and iterate(K=0) == 0
    # dimensions that do not match the system
    P.na = 3
    assert init() == E_SIZE and iterate() == E_SIZE
    P.na = 2
    # an unknown system
    P.system = 9
    assert init() == E_SYSTEM and iterate() == E_SYSTEM
