"""NN(..., deterministic=True): the gradients of the 'sine' critic and its actor with fixed-order sums (cacto_*_grad_det).  The same
inputs must give the same bits run after run -- also while another stream keeps the GPU busy, so that the CTAs start and finish in
a different order -- through the eager update, the captured and the pipelined update graphs, learn_and_update with both buffers,
simulated data-parallel ranks and one all-GPU episode.  The results agree with the default (atomic) path up to summation order."""
import os
import random
import subprocess
import sys

import numpy as np
import pytest
import torch

from cacto_b200.conf import get_conf
from test_gpu_nn import rel
from test_gpu_update_graph import fill

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def make(system, B, deterministic=True, seed=0, w_S=1e-2, engine='auto', **over):
    from cacto_b200 import environment as genv
    from cacto_b200.NeuralNetwork import NN
    from cacto_b200.RL import RL_AC
    conf = get_conf(system, **over)
    env = genv.make_env(conf)
    nn = NN(env, conf, w_S, seed=seed, deterministic=deterministic)
    nn.update_engine = engine
    rl = RL_AC(env, nn, conf, 0)
    rl.setup_model()
    rng = np.random.default_rng(seed + 1)
    ns = conf.nb_state
    lo, hi = np.asarray(conf.x_init_min, float), np.asarray(conf.x_init_max, float)
    f = lambda a, dt=torch.float32: torch.tensor(np.asarray(a), dtype=dt, device='cuda')
    dv = rng.normal(size=(B, ns))
    dv[:, -1] = 0
    batch = (f(rng.uniform(lo, hi, (B, ns))), f(rng.uniform(-5, 0, (B, 1))), f(rng.uniform(lo, hi, (B, ns))), f(dv),
             f(rng.uniform(size=(B, 1)) < 0.5), f(rng.uniform(size=(B, 1)) < 0.2, torch.float64), f(rng.uniform(0.2, 1.5, (B, 1))))
    return conf, nn, rl, batch


def grads(nn, rl, batch):
    s, pr, sn, dv, d, term, w = batch
    _, rtg, V, Vt = nn.compute_critic_grad(rl.critic_model, rl.target_critic, s, sn, pr, dv, d, w)
    out = dict(critic=rl.critic_model.grad.clone(), rtg=rtg.clone(), V=V.clone(), Vt=Vt.clone(), loss=nn.last_critic_loss.clone())
    _, act = nn.compute_actor_grad(rl.actor_model, rl.critic_model, s, term, None, return_actions=True)
    out.update(actor=rl.actor_model.grad.clone(), act=act.clone())
    torch.cuda.synchronize()
    return out


def busy_gpu():
    """A benign load on a side stream (a chain of large matmuls) that runs beside the next launches of the current stream."""
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        a = torch.randn(6144, 6144, device='cuda') / 80.0
        for _ in range(24):
            a = torch.tanh(a @ a)
    return side, a


GRAD_CASES = [('manipulator', 64, {}), ('manipulator', 500, {}), ('manipulator', 2000, {}),
              ('manipulator', 4096, {}), ('manipulator', 3000, dict(w_S=0.0)), ('ur5', 2304, {}), ('car', 16384, {}),   # tcgen05 engine
              ('manipulator', 4096, dict(engine='fma')),
              ('manipulator', 16384, dict(engine='fma')),       # 1024 tiles: four waves over the 296 slices
              ('manipulator', 64, dict(NH1=128, NH2=128)), ('manipulator', 4096, dict(NH1=128, NH2=128)),
              ('car', 64, {}), ('ur5', 64, {}), ('manipulator', 128, dict(MC=1))]


@pytest.mark.parametrize('system,B,over', GRAD_CASES)
def test_gradients_are_bit_identical_run_to_run(system, B, over):
    conf, nn, rl, batch = make(system, B, **over)
    assert nn._use_tc(B) == (B >= nn.TC_MIN_BATCH and over.get('engine') != 'fma')
    a = grads(nn, rl, batch)
    side, keep = busy_gpu()
    b = grads(nn, rl, batch)
    side.synchronize()
    c = grads(nn, rl, batch)
    for k in a:
        assert torch.equal(a[k], b[k]), k
        assert torch.equal(a[k], c[k]), k
    assert float(a['loss']) > 0 and torch.isfinite(a['critic']).all() and torch.isfinite(a['actor']).all()


@pytest.mark.parametrize('system,B,over', GRAD_CASES)
def test_gradients_match_the_default_path(system, B, over):
    """Same weights (same seed), same batch: the two paths differ only in the order of the sums."""
    _, nn_d, rl_d, batch = make(system, B, **over)
    _, nn_a, rl_a, _ = make(system, B, deterministic=False, **over)
    a, b = grads(nn_d, rl_d, batch), grads(nn_a, rl_a, batch)
    for k in ('rtg', 'V', 'Vt', 'act'):
        assert torch.equal(a[k], b[k]), k         # per-sample outputs: no cross-CTA sums
    tol = 1e-5 if B < 8192 else 2e-5
    assert rel(a['critic'], b['critic'].cpu().numpy()) < tol
    assert rel(a['actor'], b['actor'].cpu().numpy()) < tol
    assert abs(float(a['loss']) - float(b['loss'])) <= 1e-5 * abs(float(b['loss']))


@pytest.mark.parametrize('system,B', [('manipulator', 64), ('car', 64), ('ur5', 19), ('manipulator', 2500)])
def test_gradients_match_the_oracle(system, B):
    """The deterministic gradients within the oracle tolerances of test_gpu_nn.py (oracle/nn.py, torch-CPU autograd)."""
    from oracle import nn as onn
    from oracle import systems as osys
    from test_gpu_nn import make as make_np
    conf, env, nn, rl, (s, pr, sn, dv, d, term, w) = make_np(system, B)
    nn.deterministic = True
    critic, target, actor = rl.critic_model.get_weights(), rl.target_critic.get_weights(), rl.actor_model.get_weights()
    target = [t + 0.01 * np.random.default_rng(5).normal(size=t.shape).astype(np.float32) for t in target]
    rl.target_critic.set_weights(target)
    cg, rtg, V, Vt, loss = onn.critic_grad(critic, target, conf, 1e-2, s, sn, pr, dv, d, w)
    g, g_rtg, g_V, g_Vt = nn.compute_critic_grad(rl.critic_model, rl.target_critic, s, sn, pr, dv, d, w)
    assert rel(g_rtg, rtg) < 2e-5 and rel(g_V, V) < 2e-5 and rel(g_Vt, Vt) < 2e-5
    assert abs(float(nn.last_critic_loss) - loss) <= 1e-4 * abs(loss)
    for gv, rv in zip(g, cg):
        assert rel(gv, rv) < 1e-4
    ag, actions, _, _ = onn.actor_grad(actor, critic, conf, osys.make_env(conf), s, term)
    ga, act = nn.compute_actor_grad(rl.actor_model, rl.critic_model, s, term, None, return_actions=True)
    assert rel(act, actions) < 2e-5
    for gv, rv in zip(ga, ag):
        assert rel(gv, rv) < 1e-4
    assert set(nn._det_ws) == ({nn.DET_CRITIC_TC, nn.DET_ACTOR_TC} if B >= nn.TC_MIN_BATCH else {nn.DET_CRITIC, nn.DET_ACTOR})


def state_of(rl):
    out = [n.params.clone() for n in (rl.critic_model, rl.target_critic, rl.actor_model)]
    out += [n.params_T.clone() for n in (rl.critic_model, rl.actor_model) if n.params_T is not None]
    for o in (rl.critic_optimizer, rl.actor_optimizer):
        out += [t.clone() for st in o._state.values() for t in st]
    return out


def same_bits(a, b):
    """Bit-for-bit equality (NaN padding included, which torch.equal would call unequal)."""
    ity = {torch.float64: torch.int64, torch.float32: torch.int32}
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.view(ity.get(a.dtype, a.dtype)), b.view(ity.get(b.dtype, b.dtype)))


def assert_same_state(x, y):
    assert len(x) == len(y)
    for i, (a, b) in enumerate(zip(x, y)):
        assert same_bits(a, b), i


UPDATE_CASES = [('manipulator', {}), ('manipulator', dict(LR_SCHEDULE=1)), ('manipulator', dict(MC=1)), ('ur5', {}),
                ('manipulator', dict(NH1=128, NH2=128))]


@pytest.mark.parametrize('system,over', UPDATE_CASES)
def test_updates_are_bit_identical(system, over):
    """Two fresh seeded RL_ACs: 10 eager updates, then 10 replays of the update graph, give the same weights and Adam moments;
    the pipelined graph after flush() equals the sequential graph."""
    from cacto_b200.replay_buffer import ReplayBuffer
    runs = []
    for run in range(2):
        conf, nn, rl, _ = make(system, 64, **over)
        buf = ReplayBuffer(conf)
        fill(buf, conf, 3000)
        side = keep = None
        if run == 1:
            side, keep = busy_gpu()
        for it in range(10):
            b = buf.sample(np.random.default_rng(it).integers(0, 3000, conf.BATCH_SIZE))
            rl.update(b[0], b[2], b[1], b[3], b[4], b[5], b[6], fuse_target=True)
        g = rl.make_update_graph()
        for it in range(10):
            buf.sample(np.random.default_rng(100 + it).integers(0, 3000, conf.BATCH_SIZE), out=g.io)
            g.replay()
        torch.cuda.synchronize()
        runs.append((state_of(rl), g.io['V'].clone(), float(nn.last_critic_loss)))
    assert_same_state(runs[0][0], runs[1][0])
    assert torch.equal(runs[0][1], runs[1][1]) and runs[0][2] == runs[1][2]
    # pipelined vs sequential graph: every kernel sees the same inputs
    out = []
    for pipelined in (False, True):
        conf, nn, rl, _ = make(system, 64, **over)
        buf = ReplayBuffer(conf)
        fill(buf, conf, 3000)
        g = rl.make_pipelined_update_graph() if pipelined else rl.make_update_graph()
        for it in range(7):
            buf.sample(np.random.default_rng(it).integers(0, 3000, conf.BATCH_SIZE), out=g.io)
            g.replay()
        if pipelined:
            g.flush()
        torch.cuda.synchronize()
        out.append(state_of(rl))
    assert_same_state(out[0], out[1])


@pytest.mark.parametrize('alpha', [0, 0.6])
def test_learn_and_update_is_bit_identical(alpha):
    from cacto_b200.replay_buffer import PrioritizedReplayBuffer, ReplayBuffer
    runs = []
    for run in range(2):
        conf, nn, rl, _ = make('manipulator', 64, prioritized_replay_alpha=alpha, UPDATE_LOOPS=np.array([12]), save_interval=10 ** 9)
        buf = PrioritizedReplayBuffer(conf) if alpha else ReplayBuffer(conf)
        fill(buf, conf, 3000)
        random.seed(0)
        np.random.seed(0)
        rl.use_update_graph = False
        cnt = rl.learn_and_update(0, buf, 0)
        rl.use_update_graph = True
        rl.learn_and_update(cnt, buf, 0)
        torch.cuda.synchronize()
        trees = [buf.storage_mat.clone()]
        if alpha:
            trees += [buf._it_sum._value.clone(), buf._it_min._value.clone()]
            assert buf._max_priority >= 1.0
        runs.append((state_of(rl), trees, getattr(buf, '_max_priority', 1.0)))
    assert_same_state(runs[0][0], runs[1][0])
    assert_same_state(runs[0][1], runs[1][1])
    assert runs[0][2] == runs[1][2]


def test_partials_stay_inside_their_workspace():
    """The kernels write only the slices the size query counts: canary bands around the workspace, the gradient blocks and the
    per-sample outputs survive a ragged batch of several waves."""
    from cacto_b200.ops import ops
    conf, nn, rl, batch = make('manipulator', 16384 - 5)
    s, pr, sn, dv, d, term, w = batch
    B, G = s.shape[0], 4096

    def guarded(n):
        big = torch.full((n + 2 * G,), 7.25, dtype=torch.float32, device='cuda')
        return big, big[G:G + n]

    def intact(big, n):
        return bool((big[:G] == 7.25).all()) and bool((big[G + n:] == 7.25).all())

    nc, na = rl.critic_model.n, rl.actor_model.n
    ns, nact = conf.nb_state, conf.nb_action
    from cacto_b200._lib import lib
    nw = int(lib.cacto_actor_width_param_count(ns, nact, 128, 96))
    sizes = dict(pc=int(ops.det_partials_floats(0, B, ns, nact, 0, 0)), pa=int(ops.det_partials_floats(1, B, ns, nact, 0, 0)),
                 pw=int(ops.det_partials_floats(2, B, ns, nact, 128, 96)), ptc=int(ops.det_partials_floats(3, B, ns, nact, 0, 0)),
                 pta=int(ops.det_partials_floats(4, B, ns, nact, 0, 0)), gc=nc, ga=na, gw=nw, gtc=nc, gta=na, rtg=B, V=B, Vt=B, loss=1,
                 act=B * nact, actw=B * nact)
    bufs = {k: guarded(n) for k, n in sizes.items()}
    for k in ('gc', 'ga', 'gw', 'gtc', 'gta', 'loss'):
        bufs[k][1].zero_()
    x = {k: v[1] for k, v in bufs.items()}
    ops.critic_grad_det(nn._pt, rl.critic_model.params, rl.critic_model.params_T, rl.target_critic.params, 1e-2, 0, s, sn, pr.reshape(-1), dv,
                        d.reshape(-1), w.reshape(-1), 1.0 / B, x['gc'], x['rtg'], x['V'], x['Vt'], x['loss'], x['pc'])
    ops.actor_grad_det(nn._pt, rl.actor_model.params, rl.actor_model.params_T, rl.critic_model.params, rl.critic_model.params_T, s, term.reshape(-1),
                       1.0 / B, x['ga'], x['act'], x['pa'])
    aw = torch.randn(nw, device='cuda') * 0.05
    ops.actor_grad_width_det(nn._pt, aw, 128, 96, rl.critic_model.params, rl.critic_model.params_T, s, term.reshape(-1), 1.0 / B, x['gw'], x['actw'],
                             x['pw'])
    ws = nn._tc_workspace(B)
    ops.critic_grad_tc_det(nn._pt, rl.critic_model.params, rl.target_critic.params, 1e-2, 0, s, sn, pr.reshape(-1), dv, d.reshape(-1), w.reshape(-1),
                           1.0 / B, x['gtc'], x['rtg'], x['V'], x['Vt'], x['loss'], ws, x['ptc'])
    ops.actor_grad_tc_det(nn._pt, rl.actor_model.params, rl.critic_model.params, s, term.reshape(-1), 1.0 / B, x['gta'], x['act'], ws, x['pta'])
    torch.cuda.synchronize()
    for k, (big, v) in bufs.items():
        assert intact(big, v.numel()), k
    nn.update_engine = 'fma'
    ref = grads(nn, rl, batch)
    assert torch.equal(x['gc'], ref['critic']) and torch.equal(x['ga'], ref['actor'])
    nn.update_engine = 'tc'
    ref = grads(nn, rl, batch)
    assert torch.equal(x['gtc'], ref['critic']) and torch.equal(x['gta'], ref['actor'])
    assert torch.isfinite(x['gw']).all()


def test_simulated_ranks_are_bit_identical():
    """Two simulated peer-memory ranks (world 2, the static launch sequence of the update graph), run twice in a child process
    (tests/peer_sim_det_check.py): identical replicas, identical runs."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'peer_sim_det_check.py')], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert 'peer-sim-det ok' in r.stdout, r.stdout[-2000:]


def episode():
    """rollout_batch -> TO_DDP.solve_batch -> rtg_batch -> buffer.add -> learn_and_update, all on the GPU."""
    from cacto_b200 import environment as genv
    from cacto_b200.NeuralNetwork import NN
    from cacto_b200.RL import RL_AC
    from cacto_b200.TO import TO_DDP
    from cacto_b200.replay_buffer import ReplayBuffer
    conf = get_conf('manipulator', NSTEPS=30, BATCH_SIZE=16, REPLAY_SIZE=2 ** 11)
    conf.UPDATE_LOOPS = np.array([3, 3])
    conf.save_interval = 10 ** 9
    env = genv.make_env(conf)
    rl = RL_AC(env, NN(env, conf, 1e-2, seed=0, deterministic=True), conf, 0)
    rl.setup_model()
    ddp = TO_DDP(env, conf)
    random.seed(3)
    np.random.seed(3)
    rng = np.random.default_rng(21)
    n = 6
    X0 = rng.uniform(np.asarray(conf.x_init_min, float), np.asarray(conf.x_init_max, float), (n, conf.nb_state))
    X0[:, -1] = conf.dt * np.round(X0[:, -1] / conf.dt)
    out = rl.rollout_batch(X0, 1)
    res = ddp.solve_batch(X0, out['states'], out['controls'], out['horizon'].cpu().numpy(), max_iter=30)
    r = rl.rtg_batch(res['TO_states'], res['TO_step_cost'])
    offs = res['offsets']
    cut = lambda t: [t.cpu().numpy()[offs[e]:offs[e + 1]] for e in range(n)]
    buf = ReplayBuffer(conf)
    buf.add(res['TO_states'], cut(r['partial']), cut(r['state_next']), res['dVdx_list'], cut(r['done']), cut(r['term']))
    assert rl.learn_and_update(0, buf, 1) == 3
    torch.cuda.synchronize()
    return state_of(rl), buf.storage_mat.clone(), res['controls'].clone()


def test_one_all_gpu_episode_is_bit_identical():
    a = episode()
    b = episode()
    assert same_bits(a[2], b[2]), 'TO solutions differ'
    assert same_bits(a[1], b[1]), 'replay storage differs'
    assert_same_state(a[0], b[0])
