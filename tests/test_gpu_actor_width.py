"""The actor at any hidden width (conf.NH1 / conf.NH2 other than 256: csrc/actor_width.cu) through every layer that uses it:
rollouts, NN.eval, the actor gradient, the update (eager, graph, pipelined graph), host transfers, plots and checkpoints, against
the oracle and, at 256, against the fused kernels."""
import random

import numpy as np
import pytest
import torch

from cacto_b200.conf import SYSTEM_IDS, get_conf
from oracle import backward as obw
from oracle import nn as onn
from oracle import per as oper
from oracle import rtg as ortg
from oracle import systems as osys

pytestmark = pytest.mark.gpu

WIDTHS = [(64, 64), (37, 100), (128, 256), (512, 512)]


def rel(a, b):
    a = a.detach().cpu().double().numpy() if isinstance(a, torch.Tensor) else np.asarray(a, dtype=float)
    b = b.detach().cpu().double().numpy() if isinstance(b, torch.Tensor) else np.asarray(b, dtype=float)
    assert a.shape == b.shape, (a.shape, b.shape)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def setup(system, widths, seed=0, w_S=1e-2, **over):
    from cacto_b200 import environment as genv
    from cacto_b200.NeuralNetwork import NN
    from cacto_b200.RL import RL_AC
    conf = get_conf(system, NH1=widths[0], NH2=widths[1], **over)
    env = genv.make_env(conf)
    nn = NN(env, conf, w_S, seed=seed)
    rl = RL_AC(env, nn, conf, 0)
    rl.setup_model()
    return conf, env, nn, rl


def ics(conf, B, seed):
    rng = np.random.default_rng(seed)
    x = rng.uniform(np.asarray(conf.x_init_min, float), np.asarray(conf.x_init_max, float), (B, conf.nb_state))
    x[:, -1] = conf.dt * np.round(x[:, -1] / conf.dt)
    return x


def batch(conf, B, seed=1):
    rng = np.random.default_rng(seed)
    ns = conf.nb_state
    lo, hi = np.asarray(conf.x_init_min, float), np.asarray(conf.x_init_max, float)
    s = rng.uniform(lo, hi, (B, ns)).astype(np.float32)
    sn = rng.uniform(lo, hi, (B, ns)).astype(np.float32)
    pr = rng.uniform(-5, 0, (B, 1)).astype(np.float32)
    dv = rng.normal(size=(B, ns)).astype(np.float32)
    dv[:, -1] = 0
    d = (rng.uniform(size=(B, 1)) < 0.5).astype(np.float32)
    term = (rng.uniform(size=(B, 1)) < 0.3).astype(np.float64)
    w = rng.uniform(0.2, 1.5, (B, 1)).astype(np.float32)
    return s, pr, sn, dv, d, term, w


# ---------------------------------------------------------------------------------------------------------------- rollouts
@pytest.mark.parametrize('widths', WIDTHS)
@pytest.mark.parametrize('system', SYSTEM_IDS)
def test_rollouts_match_oracle(system, widths):
    conf, env, nn, rl = setup(system, widths)
    assert rl.actor_model.kind == 'actor_width' and rl.actor_model.params_T is None
    B = 70 if system != 'ur5' else 37                  # more than one 32-rollout CTA, ragged last tile
    X0 = ics(conf, B, 3)
    X0[0, -1] = 0.0                                    # full horizon
    X0[1, -1] = (conf.NSTEPS - 1) * conf.dt            # one step
    X0[2, -1] = conf.NSTEPS * conf.dt                  # zero horizon
    out = rl.rollout_batch(X0, 1, with_reward=True)    # rollout_engine 'tc' (the default) is ignored for this actor
    states = out['states'].permute(2, 0, 1).cpu().numpy()
    controls = out['controls'].permute(2, 0, 1).cpu().numpy()
    rewards = out['rewards'].cpu().numpy()
    hz = out['horizon'].cpu().numpy()
    assert out['success'].cpu().numpy().all()
    oenv = osys.make_env(conf)
    ap = onn.to_torch(rl.actor_model.get_weights())

    def actor_eval(x):
        with torch.no_grad():
            return onn.actor_forward(ap, torch.tensor(x, dtype=torch.float32), conf).numpy()[0]
    check = [0, 1, 2, 31, 32, B - 1] if system != 'ur5' else [0, 1, 2, B - 1]
    for b in check:
        T = ortg.horizon(conf, X0[b, -1])
        assert T == hz[b]
        assert np.isnan(states[b, T + 1:]).all() and np.isnan(controls[b, T:]).all()      # past the horizon: untouched
        if T == 0:
            assert np.array_equal(states[b, 0], X0[b]) and np.isnan(rewards[:, b]).all()
            continue
        _, st, ct, T_o, ok = ortg.create_to_init(conf, oenv, actor_eval, 1, X0[b])
        assert ok == 1 and T_o == T
        sc = np.abs(st).max(axis=0) + 1e-12
        assert (np.abs(states[b, :T + 1] - st) / sc).max() < 1e-4, (b, T)
        assert np.abs(controls[b, :T] - ct).max() <= 1e-4 * max(np.abs(ct).max(), 1e-3)
        if system != 'ur5':        # UR5: the rollout reward is Env.step's bounded control cost, env.reward's is u.u (quirk Q8)
            r = [oenv.reward(conf.cost_weights_running, states[b, k], controls[b, k]) for k in range(T)]
            r.append(oenv.reward(conf.cost_weights_terminal, states[b, T]))
            np.testing.assert_allclose(rewards[:T + 1, b], r, rtol=1e-6, atol=1e-9)


def test_nan_initial_state_fails_the_rollout():
    conf, env, nn, rl = setup('car', (37, 100))
    X0 = ics(conf, 40, 5)
    X0[0, -1] = 0.0
    X0[3, 0] = np.nan
    out = rl.rollout_batch(X0, 1)
    fl = out['success'].cpu().numpy()
    assert fl[3] == 0 and fl[np.arange(40) != 3].all()


def test_width_kernel_agrees_with_fma_engine_at_256():
    """The width-generic rollout op on a 256-wide actor against the fused 'fma' engine on the same actor."""
    from cacto_b200.ops import ops
    conf, env, nn, rl = setup('manipulator', (256, 256))
    am = rl.actor_model
    assert am.kind == 'actor'
    B, T, ns, na = 40000, conf.NSTEPS, conf.nb_state, conf.nb_action
    X0 = ics(conf, B, 7)
    ref = rl.rollout_batch(X0, 1, engine='fma')
    dev = am.params.device
    icsd = torch.as_tensor(X0, device=dev)
    hz = ref['horizon']
    assert len(np.unique(hz.cpu().numpy())) > 10                         # mixed horizons

    def run():
        st = torch.full((T + 1, ns, B), float('nan'), dtype=torch.float64, device=dev)
        ct = torch.full((T, na, B), float('nan'), dtype=torch.float64, device=dev)
        fl = torch.empty(B, dtype=torch.int32, device=dev)
        ops.rollout_width(env._pt, am.params, 256, 256, icsd, hz, T, st, ct, fl, None)
        return st, ct, fl
    st, ct, fl = run()
    assert torch.equal(fl, ref['success'])
    assert torch.equal(torch.isnan(st), torch.isnan(ref['states'])) and torch.equal(torch.isnan(ct), torch.isnan(ref['controls']))
    m = ~torch.isnan(st)
    sc = ref['states'].abs().nan_to_num(0).amax(dim=(0, 2), keepdim=True) + 1e-12
    assert float(((st - ref['states']).abs() / sc)[m].max()) < 1e-5
    mc = ~torch.isnan(ct)
    assert float((ct - ref['controls']).abs()[mc].max()) < 1e-5
    st2, ct2, fl2 = run()
    assert torch.equal(st2.nan_to_num(7.0), st.nan_to_num(7.0)) and torch.equal(ct2.nan_to_num(7.0), ct.nan_to_num(7.0)) and torch.equal(fl2, fl)


def test_host_paths_deliver_the_rollout_batch_knots():
    from cacto_b200.RL import CompactRollouts
    conf, env, nn, rl = setup('manipulator', (128, 64))
    B, T, ns, na = 700, conf.NSTEPS, conf.nb_state, conf.nb_action
    X0 = ics(conf, B, 11)
    ih = torch.as_tensor(X0).pin_memory()
    ref = rl.rollout_batch(X0, 1)
    hz = ref['horizon'].cpu().numpy()
    rs, rc = ref['states'].cpu().numpy(), ref['controls'].cpu().numpy()
    knots = np.broadcast_to((np.arange(T + 1)[:, None] <= hz[None, :])[:, None, :], rs.shape)
    cknots = np.broadcast_to((np.arange(T)[:, None] < hz[None, :])[:, None, :], rc.shape)
    for mode in ('pipelined', 'zero_copy', 'staged'):
        st = torch.full((T + 1, ns, B), float('nan'), dtype=torch.float64).pin_memory()
        ct = torch.full((T, na, B), float('nan'), dtype=torch.float64).pin_memory()
        fl = torch.zeros(B, dtype=torch.int32).pin_memory()
        h = rl.rollout_to_host(ih, 1, st, ct, fl, mode=mode, n_chunks=3)
        assert (h == hz).all() and bool(fl.all()), mode
        assert np.array_equal(st.numpy()[knots], rs[knots]), mode            # the same kernel on the same rollouts: same bits
        assert np.array_equal(ct.numpy()[cknots], rc[cknots]), mode
    st = torch.full((T + 1, ns - 1, B), float('nan'), dtype=torch.float64).pin_memory()
    ct = torch.full((T, na, B), float('nan'), dtype=torch.float32).pin_memory()
    fl = torch.zeros(B, dtype=torch.int32).pin_memory()
    h = rl.rollout_to_host(ih, 1, st, ct, fl, compact=True, n_chunks=3)
    assert np.array_equal(st.numpy()[knots[:, :ns - 1]], rs[:, :ns - 1][knots[:, :ns - 1]])
    assert np.array_equal(ct.numpy().astype(np.float64)[cknots], rc[cknots])
    assert CompactRollouts is not None and bool(fl.all())


def test_plot_rollout_runs_with_a_narrow_actor(capsys):
    from cacto_b200.plot_utils import PLOT
    conf, env, nn, rl = setup('manipulator', (64, 64), seed=3)
    init = ics(conf, 4, 4)
    init[:, -1] = 0.0
    plot = PLOT(7, env, nn, conf)
    returns = plot.rollout(123, rl.actor_model, init)
    assert len(returns) == 4 and all(np.isfinite(v) for v in returns.values())
    ref = rl.rollout_batch(init, 1)
    np.testing.assert_array_equal(plot.rollout_states, ref['states'].permute(2, 0, 1).cpu().numpy())


# ---------------------------------------------------------------------------------------------------------------- NN
@pytest.mark.parametrize('widths', [(37, 100), (512, 512)])
def test_eval_matches_oracle(widths):
    conf, env, nn, rl = setup('ur5', widths)
    s = batch(conf, 77)[0]
    got = nn.eval(rl.actor_model, s)
    ref = onn.actor_forward(onn.to_torch(rl.actor_model.get_weights()), torch.as_tensor(s), conf)
    assert rel(got, ref) < 2e-6


@pytest.mark.parametrize('system,B,widths', [(sy, B, wd) for sy in ('manipulator', 'car', 'ur5') for B in (1, 19, 64)
                                             for wd in ((128, 64), (37, 100), (512, 512))] +
                         [('manipulator', 4096, (128, 64)), ('car', 4096, (37, 100)), ('ur5', 4096, (512, 512))])
def test_actor_gradient_matches_oracle(system, B, widths):
    conf, env, nn, rl = setup(system, widths)
    s, pr, sn, dv, d, term, w = batch(conf, B)
    actor, critic = rl.actor_model.get_weights(), rl.critic_model.get_weights()
    oenv = osys.PooledEnv(osys.make_env(conf)) if B > 1000 else osys.make_env(conf)
    ag, actions, s_next, dQ = onn.actor_grad(actor, critic, conf, oenv, s, term)
    ga, act = nn.compute_actor_grad(rl.actor_model, rl.critic_model, s, term, None, return_actions=True)
    assert rel(act, actions) < 2e-5
    for k, (gv, rv) in enumerate(zip(ga, ag)):
        assert rel(gv, rv) < 1e-4, k


@pytest.mark.parametrize('B', [19, 4096])
def test_width_op_agrees_with_fused_actor_gradient_at_256(B):
    from cacto_b200.ops import ops
    conf, env, nn, rl = setup('manipulator', (256, 256))
    am, cm = rl.actor_model, rl.critic_model
    s, pr, sn, dv, d, term, w = batch(conf, B)
    st = torch.as_tensor(s, device=am.params.device)
    tm = torch.as_tensor(term, device=am.params.device).reshape(-1)
    nn.update_engine = 'fma'
    ref = [g.clone() for g in nn.compute_actor_grad(am, cm, s, term, None)]
    am.grad.zero_()
    acts = torch.empty((B, am.na), dtype=torch.float32, device=st.device)
    ops.actor_grad_width(env._pt, am.params, 256, 256, cm.params, cm.params_T, st, tm, 1.0 / B, am.grad, acts)
    for gv, rv in zip(am._grad_views, ref):
        assert rel(gv, rv) <= 2e-5
    torch.testing.assert_close(acts, nn.eval(am, s), rtol=0, atol=1e-6)


def test_shard_gradients_sum_to_the_full_batch_gradient():
    conf, env, nn, rl = setup('car', (37, 100))
    B = 1000
    s, pr, sn, dv, d, term, w = batch(conf, B)
    full = [g.clone() for g in nn.compute_actor_grad(rl.actor_model, rl.critic_model, s, term, None)]
    acc = [torch.zeros_like(g) for g in full]
    for lo, hi in ((0, 300), (300, 301), (301, 1000)):
        part = nn.compute_actor_grad(rl.actor_model, rl.critic_model, s[lo:hi], term[lo:hi], None, global_batch=B)
        for a, p in zip(acc, part):
            a += p
    for a, f in zip(acc, full):
        assert rel(a, f) <= 2e-5


@pytest.mark.parametrize('critic_type', ['relu', 'elu'])
def test_critic_variant_with_a_narrow_actor(critic_type):
    conf, env, nn, rl = setup('manipulator', (128, 64), critic_type=critic_type)
    assert rl.critic_model.kind == 'critic_generic' and rl.actor_model.kind == 'actor_width'
    s, pr, sn, dv, d, term, w = batch(conf, 19)
    ag = onn.actor_grad(rl.actor_model.get_weights(), rl.critic_model.get_weights(), conf, osys.make_env(conf), s, term)[0]
    for gv, rv in zip(nn.compute_actor_grad(rl.actor_model, rl.critic_model, s, term, None), ag):
        assert rel(gv, rv) < 1e-4


def test_generic_critic_path_admits_a_512_wide_actor():
    conf, env, nn, rl = setup('car', (512, 512), critic_type='elu')
    s, pr, sn, dv, d, term, w = batch(conf, 5)
    ag = onn.actor_grad(rl.actor_model.get_weights(), rl.critic_model.get_weights(), conf, osys.make_env(conf), s, term)[0]
    for gv, rv in zip(nn.compute_actor_grad(rl.actor_model, rl.critic_model, s, term, None), ag):
        assert rel(gv, rv) < 1e-4


def test_relu_critic_refuses_widths_beyond_its_kernels():
    with pytest.raises(ValueError, match='relu'):
        setup('car', (512, 64), critic_type='relu')


# ---------------------------------------------------------------------------------------------------------------- update
@pytest.mark.parametrize('system,widths', [('manipulator', (128, 64)), ('ur5', (37, 100))])
def test_two_update_steps_match_oracle(system, widths):
    conf, env, nn, rl = setup(system, widths)
    s, pr, sn, dv, d, term, w = batch(conf, 64)
    critic, target, actor = rl.critic_model.get_weights(), rl.target_critic.get_weights(), rl.actor_model.get_weights()
    oc, oa = onn.Adam(critic, conf.CRITIC_LEARNING_RATE), onn.Adam(actor, conf.ACTOR_LEARNING_RATE)
    oenv = osys.make_env(conf)
    for step in range(2):
        out = onn.update(critic, target, actor, oc, oa, conf, 1e-2, oenv, (s, pr, sn, dv, d, term, w))
        rtg, V, Vt = rl.update(s, sn, pr, dv, d, term, w)
        rl.update_target(rl.target_critic.variables, rl.critic_model.variables)
        assert rel(rtg, out['rtg']) < 2e-5 and rel(V, out['V']) < 2e-5
        for k, (m, r) in enumerate(zip(rl.critic_model.get_weights() + rl.actor_model.get_weights(), critic + actor)):
            assert rel(m, r) < 1e-4, (step, k)


def _fill(buffer, conf, n_rows, seed=0):
    rng = np.random.default_rng(seed)
    ns = conf.nb_state
    lo, hi = np.asarray(conf.x_init_min, float), np.asarray(conf.x_init_max, float)
    dv = rng.normal(size=(n_rows, ns))
    dv[:, -1] = 0
    buffer.add((rng.uniform(lo, hi, (n_rows, ns)),), (rng.uniform(-5, 0, n_rows),), (rng.uniform(lo, hi, (n_rows, ns)),), (dv,),
               ((rng.uniform(size=n_rows) < 0.5).astype(float),), ((rng.uniform(size=n_rows) < 0.05).astype(float),))


def _weights(rl):
    return [w.copy() for n in (rl.critic_model, rl.target_critic, rl.actor_model) for w in n.get_weights()]


def test_graph_replays_equal_eager_updates_and_pipelined_graph_equals_sequential():
    from cacto_b200.replay_buffer import ReplayBuffer
    widths = (100, 37)
    conf, _, _, rl_e = setup('manipulator', widths)
    _, _, _, rl_g = setup('manipulator', widths)
    _, _, _, rl_p = setup('manipulator', widths)
    buf = ReplayBuffer(conf)
    _fill(buf, conf, 5000)
    g, gp = rl_g.make_update_graph(), rl_p.make_pipelined_update_graph()
    for it in range(5):
        idx = np.random.default_rng(it).integers(0, 5000, conf.BATCH_SIZE)
        b = buf.sample(idx)
        rtg_e, V_e, _ = rl_e.update(b[0], b[2], b[1], b[3], b[4], b[5], b[6], fuse_target=True)
        buf.sample(idx, out=g.io)
        rtg_g, V_g, _ = g.replay()
        buf.sample(idx, out=gp.io)
        gp.replay()
        torch.testing.assert_close(rtg_g, rtg_e, rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(V_g, V_e, rtol=1e-5, atol=1e-6)
    gp.flush()
    for a, b_, c in zip(_weights(rl_e), _weights(rl_g), _weights(rl_p)):
        assert np.abs(a - b_).max() <= 2e-5 * max(np.abs(a).max(), 1e-3)
        assert np.abs(c - b_).max() <= 2e-5 * max(np.abs(b_).max(), 1e-3)


def test_large_batch_update_runs_tc_critic_and_width_actor():
    conf, env, nn, rl = setup('manipulator', (128, 64), BATCH_SIZE=4096)
    assert nn.update_engine == 'auto' and nn._use_tc(4096)
    s, pr, sn, dv, d, term, w = batch(conf, 4096)
    actor, critic = rl.actor_model.get_weights(), rl.critic_model.get_weights()
    ag = onn.actor_grad(actor, critic, conf, osys.PooledEnv(osys.make_env(conf)), s, term)[0]
    for gv, rv in zip(nn.compute_actor_grad(rl.actor_model, rl.critic_model, s, term, None), ag):
        assert rel(gv, rv) < 1e-4
    before = rl.actor_model.get_weights()
    rl.update(s, sn, pr, dv, d, term, w)
    torch.cuda.synchronize()
    after = rl.actor_model.get_weights()
    assert all(np.isfinite(a).all() for a in after) and any(not np.array_equal(a, b) for a, b in zip(after, before))


# ---------------------------------------------------------------------------------------------------------------- checkpoints
@pytest.mark.parametrize('ext', ['.h5', '.npz'])
def test_checkpoint_round_trip(tmp_path, ext):
    conf, env, nn, rl = setup('car', (100, 37))
    w0 = [x + 0.1 * np.random.default_rng(1).normal(size=x.shape).astype(np.float32) for x in rl.actor_model.get_weights()]
    rl.actor_model.set_weights(w0)
    path = str(tmp_path / ('actor' + ext))
    rl.actor_model.save_weights(path)
    _, _, _, rl2 = setup('car', (100, 37), seed=9)
    rl2.actor_model.load_weights(path)
    for a, b in zip(rl2.actor_model.get_weights(), w0):
        assert a.dtype == b.dtype and np.array_equal(a, b)
    s = batch(conf, 9)[0]
    assert torch.equal(rl2.NN.eval(rl2.actor_model, s), nn.eval(rl.actor_model, s))


def test_loading_a_256_wide_file_into_a_128_wide_actor_raises(tmp_path):
    _, _, _, rl = setup('car', (256, 256))
    path = str(tmp_path / 'actor.h5')
    rl.actor_model.save_weights(path)
    _, _, _, rl2 = setup('car', (128, 128))
    before = rl2.actor_model.get_weights()
    with pytest.raises(AssertionError, match=r'256\).*128\)'):           # Network.set_weights: (file shape, actor shape)
        rl2.actor_model.load_weights(path)
    for a, b in zip(rl2.actor_model.get_weights(), before):                # refused before any layer was written
        assert np.array_equal(a, b)


# ---------------------------------------------------------------------------------------------------------------- training loop
def _draw_ics(conf, B, seed):
    rng = np.random.default_rng(seed)
    x = rng.uniform(np.asarray(conf.x_init_min, float), np.asarray(conf.x_init_max, float), (B, conf.nb_state))
    x[:, -1] = conf.dt * np.round(x[:, -1] / conf.dt)
    x[0, -1] = 0.0
    return x


@pytest.mark.parametrize('system,alpha', [('single_integrator', 0.6), ('car', 0.0), ('manipulator', 0.0)])
def test_two_episodes_of_the_training_loop_match_the_oracle_with_a_narrow_actor(system, alpha):
    """The harness of tests/test_gpu_pipeline.py with a (128, 64) actor: rollouts, updates (graph, pipelined) and PER on the
    width-generic kernels, episode 1 rolling out the updated narrow actor."""
    from cacto_b200 import environment as genv
    from cacto_b200.NeuralNetwork import NN
    from cacto_b200.RL import RL_AC
    from cacto_b200.TO import TO_Casadi
    from cacto_b200.replay_buffer import PrioritizedReplayBuffer, ReplayBuffer
    over = dict(BATCH_SIZE=16, REPLAY_SIZE=2 ** 11, prioritized_replay_alpha=alpha, NH1=128, NH2=64)
    if system != 'single_integrator':
        over['NSTEPS'] = 60 if system == 'car' else 30
    conf = get_conf(system, **over)
    conf.UPDATE_LOOPS = np.array([3, 3])
    conf.save_interval = 10 ** 9
    w_S, n_ics = 1e-2, 4
    env = genv.make_env(conf)
    nn = NN(env, conf, w_S, seed=0)
    rl = RL_AC(env, nn, conf, 0)
    rl.setup_model()
    assert rl.actor_model.kind == 'actor_width'
    trop = TO_Casadi(env, conf, None, w_S)
    buf = ReplayBuffer(conf) if alpha == 0 else PrioritizedReplayBuffer(conf)

    oenv = osys.make_env(conf)
    critic, target, actor = rl.critic_model.get_weights(), rl.target_critic.get_weights(), rl.actor_model.get_weights()
    oc, oa = onn.Adam(critic, conf.values_schedule_LR_C[0]), onn.Adam(actor, conf.values_schedule_LR_A[0])
    obuf = oper.ReplayBuffer(conf) if alpha == 0 else oper.PrioritizedReplayBuffer(conf)

    counter, n_rows = 0, 0
    for ep in range(2):
        X0 = _draw_ics(conf, n_ics, 10 + ep)
        # ------------------------------------------------------------------ GPU modules
        out = rl.rollout_batch(X0, ep, with_reward=True)
        assert out['success'].cpu().numpy().all()
        hz = out['horizon'].cpu().numpy()
        S = out['states'].permute(2, 0, 1).cpu().numpy()
        U = out['controls'].permute(2, 0, 1).cpu().numpy()
        R = out['rewards'].permute(1, 0).cpu().numpy()
        TO_states = [S[b, :hz[b] + 1] for b in range(n_ics)]
        TO_controls = [U[b, :hz[b]] for b in range(n_ics)]
        TO_cost = [-R[b, :hz[b] + 1] for b in range(n_ics)]
        Vx, offs = trop.backward_pass_batch(TO_states, TO_controls)
        Vx = Vx.cpu().numpy()
        r = rl.rtg_batch(TO_states, TO_cost)
        cut = lambda t: [t.cpu().numpy()[offs[e]:offs[e + 1]] for e in range(n_ics)]
        buf.add(TO_states, cut(r['partial']), cut(r['state_next']), [Vx[offs[e]:offs[e + 1]] for e in range(n_ics)], cut(r['done']), cut(r['term']))
        # ------------------------------------------------------------------ oracle modules
        ap = onn.to_torch(actor)

        def actor_eval(x):
            with torch.no_grad():
                return onn.actor_forward(ap, torch.tensor(x, dtype=torch.float32), conf).numpy()[0]
        lists = [[] for _ in range(6)]
        for b in range(n_ics):
            _, st, ct, T, ok = ortg.create_to_init(conf, oenv, actor_eval, ep, X0[b])
            assert ok == 1 and T == hz[b]
            cost = [-oenv.reward(conf.cost_weights_running, st[t], ct[t]) for t in range(T)] + [-oenv.reward(conf.cost_weights_terminal, st[T])]
            dV = obw.backward_pass(oenv, T + 1, st, ct)
            state_arr, partial, total, s_next, done, rwrd, term, ep_ret = ortg.rl_solve(conf, st, cost)
            for l, v in zip(lists, (state_arr, partial, s_next, dV, done, term)):
                l.append(v)
        obuf.add(*lists)
        # ------------------------------------------------------------------ the experiences both sides stored
        n_new = int(sum(hz + 1))
        got = buf.storage_mat[n_rows:n_rows + n_new].cpu().numpy()
        want = obuf.storage_mat[n_rows:n_rows + n_new]
        ns = conf.nb_state
        tol = 1e-9 if ep == 0 else 2e-3                        # episode 1 rolls out the actor both sides have trained (fp32, 1e-4 apart)
        assert rel(got[:, :ns], want[:, :ns]) < tol                                   # states
        assert rel(got[:, ns], want[:, ns]) < max(tol, 1e-6)                          # partial reward-to-go (float32-rounded)
        assert rel(got[:, ns + 1:2 * ns + 1], want[:, ns + 1:2 * ns + 1]) < tol       # n-step next states
        assert rel(got[:, 2 * ns + 1:3 * ns + 1], want[:, 2 * ns + 1:3 * ns + 1]) < max(tol, 1e-6) * 10   # dVdx
        assert np.array_equal(got[:, 3 * ns + 1:], want[:, 3 * ns + 1:])              # done, term
        n_rows += n_new
        assert buf.next_idx == obuf.next_idx == n_rows
        # ------------------------------------------------------------------ updates (same index draws: same seeds)
        np.random.seed(77 + ep); random.seed(78 + ep)
        counter = rl.learn_and_update(counter, buf, ep)
        np.random.seed(77 + ep); random.seed(78 + ep)
        for _ in range(int(conf.UPDATE_LOOPS[ep])):
            s_, r_, s1_, dv_, d_, term_, w_, idx_ = obuf.sample()
            o = onn.update(critic, target, actor, oc, oa, conf, w_S, oenv, (s_, r_, s1_, dv_, d_, term_, w_))
            if alpha != 0:
                obuf.update_priorities(idx_, o['rtg'], o['V'], o['V_target'])
        assert counter == 3 * (ep + 1) and rl.update_graph is not None
        wt = 2e-4 if ep == 0 else 5e-3
        for m, ref in zip(rl.critic_model.get_weights() + rl.actor_model.get_weights() + rl.target_critic.get_weights(), critic + actor + target):
            assert rel(m, ref) < wt
        if alpha != 0:
            np.testing.assert_allclose(buf._it_sum._value.cpu().numpy()[1], obuf._it_sum.val[1], rtol=1e-3 if ep == 0 else 2e-2)
