"""CPU-side checks of the drop-in boundary: libcacto_b200.so loads without a GPU, exports exactly the symbols
include/cacto_b200.h declares, the ctypes mirror of cacto_sys_params has the C layout, and bad arguments are
rejected with negative codes before anything is launched (no compute calls here)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import cacto_b200._lib as L
    hdr = open(os.path.join(ROOT, 'include', 'cacto_b200.h')).read()
    declared = set(re.findall(r'\b(cacto_[a-z0-9_]+)\s*\(', hdr))
    assert declared == set(L.EXPORTED_SYMBOLS)
    nm = subprocess.run(['nm', '-D', '--defined-only', L.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r' T (cacto_[a-z0-9_]+)', nm))
    assert declared <= exported, declared - exported
    assert L.lib.cacto_abi_version() == 1


def test_param_counts_match_survey():
    import cacto_b200._lib as L
    # SURVEY.md section 8: critic(sine) = 64 ns + 29185, actor = 256 ns + 257 na + 66048
    for ns, na in ((3, 2), (5, 2), (6, 2), (7, 3), (13, 6)):
        assert L.lib.cacto_critic_param_count(ns) == 64 * ns + 29185
        assert L.lib.cacto_actor_param_count(ns, na) == 256 * ns + 257 * na + 66048


def test_sys_params_struct_layout_matches_header(tmp_path):
    """Compile a tiny C program against the header and compare sizeof/offsetof with the ctypes mirror."""
    import cacto_b200._lib as L
    src = tmp_path / 'layout.c'
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cacto_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu\\n",'
                   'sizeof(cacto_sys_params), offsetof(cacto_sys_params, dt), offsetof(cacto_sys_params, scale),'
                   'offsetof(cacto_sys_params, w_running), offsetof(cacto_sys_params, chain), sizeof(cacto_chain));return 0;}\n')
    exe = tmp_path / 'layout'
    subprocess.run(['gcc', '-I' + os.path.join(ROOT, 'include'), str(src), '-o', str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()]
    P = L.SysParams
    assert got == [C.sizeof(P), P.dt.offset, P.scale.offset, P.w_running.offset, P.chain.offset, C.sizeof(L.Chain)]


def test_make_sys_params_packs_conf():
    import cacto_b200._lib as L
    from cacto_b200.conf import get_conf
    for sid in ('single_integrator', 'car_park', 'manipulator', 'ur5'):
        conf = get_conf(sid)
        P = L.make_sys_params(conf)
        assert (P.nx, P.ns, P.na) == (conf.nx, conf.nb_state, conf.nb_action)
        assert P.dt == conf.dt and P.scale == 1e-5 and P.offset == 0
        np.testing.assert_array_equal(list(P.state_norm)[:conf.nb_state], np.asarray(conf.state_norm_arr, float))
        np.testing.assert_array_equal(list(P.w_running)[:len(conf.cost_weights_running)], conf.cost_weights_running)
    P = L.make_sys_params(get_conf('manipulator'))
    assert P.chain.n == 3 and list(P.chain.p[0]) == [-7.0, 0.0, 0.0] and list(P.chain.p[1]) == [10.0, 0.0, 0.0]
    P = L.make_sys_params(get_conf('ur5'))
    assert P.chain.n == 6 and P.chain.mass[1] == 8.393 and list(P.chain.axis) == [2, 1, 1, 1, 2, 1]


def test_bad_arguments_are_rejected_without_launching():
    import cacto_b200._lib as L
    from cacto_b200.conf import get_conf
    lib = L.lib
    P = L.make_sys_params(get_conf('manipulator'))
    null = C.c_void_p(0)
    assert lib.cacto_dyn_step(null, 0, 0, null, null, null, 4, null) == -1            # CACTO_E_ARG
    assert lib.cacto_dyn_step(C.byref(P), 7, 0, null, null, null, 4, null) == -3      # CACTO_E_DTYPE
    assert lib.cacto_dyn_step(C.byref(P), 0, 0, null, null, null, -1, null) == -4     # CACTO_E_SIZE
    assert lib.cacto_dyn_step(C.byref(P), 0, 0, null, null, null, 0, null) == 0       # empty batch is a no-op
    P.system = 99
    assert lib.cacto_dyn_step(C.byref(P), 0, 0, null, null, null, 4, null) == -2      # CACTO_E_SYSTEM
    assert lib.cacto_segtree_update(null, null, 64, null, null, 4, null, null) == -1
    assert lib.cacto_segtree_reduce(C.c_void_p(8), null, 63, 0, 10, C.c_void_p(8), null) == -4   # capacity not a power of two
    assert lib.cacto_rtg_window(null, 1, null, null, 3, 5, 0, null, null, null, null, null, null, null) == -1
    # data-parallel entry points: peer tables and regions
    one = C.c_void_p(16)
    tbl = (C.c_void_p * 2)(16, 16)
    assert lib.cacto_adam_step_peer(null, tbl, tbl, 2, 0, null, 0, one, one, one, 0.9, 0.999, 1e-7, null, 0.0, null, 0, 7, 3, 8, 0, null) == -1
    assert lib.cacto_adam_step_peer(one, tbl, tbl, 9, 0, null, 0, one, one, one, 0.9, 0.999, 1e-7, null, 0.0, null, 0, 7, 3, 8, 0, null) == -1   # > CACTO_MAX_PEERS
    assert lib.cacto_adam_step_peer(one, tbl, tbl, 2, 2, null, 0, one, one, one, 0.9, 0.999, 1e-7, null, 0.0, null, 0, 7, 3, 8, 0, null) == -1   # rank >= world
    assert lib.cacto_adam_step_peer(one, tbl, tbl, 2, 0, null, 0, one, one, one, 0.9, 0.999, 1e-7, null, 0.0, one, 1, 7, 3, 8, 0, null) == -4    # n != critic size
    out = C.c_void_p()
    assert lib.cacto_peer_alloc(0, C.byref(out)) == -1 and lib.cacto_peer_free(null) == -1
    assert lib.cacto_peer_export(null, null) == -1 and lib.cacto_peer_open(null, C.byref(out)) == -1 and lib.cacto_peer_close(null) == -1


def test_peer_region_layout():
    """Host-side layout of the peer-memory block: two 128-byte flag rows, then 128-byte-aligned gradient blocks."""
    from cacto_b200.parallel import PeerReduce
    for nc, na in ((29377, 67330), (30017, 70918), (1, 1)):
        total = PeerReduce.region_bytes(nc, na)
        assert total % 128 == 0 and total >= 256 + 4 * (nc + na)
        assert total - (256 + 4 * (nc + na)) < 256


def test_product_path_fails_loudly_without_cuda():
    # in a child process with every GPU hidden, so that the check also runs on a machine that has one
    code = ('import numpy as np, torch\n'
            'assert not torch.cuda.is_available()\n'
            'from cacto_b200 import environment as genv\n'
            'from cacto_b200.conf import get_conf\n'
            'env = genv.make_env(get_conf("single_integrator"))\n'
            'try:\n'
            '    env.simulate_batch(np.zeros((2, 3)), np.zeros((2, 2)))\n'
            'except RuntimeError as exc:\n'
            '    print(exc)\n'
            'else:\n'
            '    raise SystemExit("simulate_batch returned without a CUDA device")\n')
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=300, cwd=ROOT,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=''))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert re.search('no CPU fallback', r.stdout), r.stdout[-2000:]
    # and nothing under cacto_b200/ may import the oracle
    for f in os.listdir(os.path.join(ROOT, 'cacto_b200')):
        if f.endswith('.py'):
            assert 'oracle' not in open(os.path.join(ROOT, 'cacto_b200', f)).read().replace('the oracle', ''), f


def test_fp16_rollout_refuses_systems_beyond_its_limits_first():
    """cacto_rollout_tc16 runs the systems with ns <= 8 and na <= 3; a UR5 parameter block is refused with CACTO_E_SYSTEM
    before any other argument is looked at, while a supported system still gets to the pointer checks."""
    import cacto_b200._lib as L
    from cacto_b200.conf import get_conf
    null = C.c_void_p(0)
    for system, code in (('ur5', -2), ('manipulator', -1)):            # CACTO_E_SYSTEM, CACTO_E_ARG
        P = L.make_sys_params(get_conf(system))
        assert L.lib.cacto_rollout_tc16(C.byref(P), null, null, null, null, 100, null, null, null, null, 64, null) == code, system
