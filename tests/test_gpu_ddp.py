"""K7 -- the batched iLQR TO solver (TO_DDP.solve_batch, csrc/ddp.cu) against its NumPy restatement (oracle/ddp.py), its invariants,
its dVdx, and one episode of the training loop with the TO solve on the GPU."""
import numpy as np
import pytest
import torch

from cacto_b200.conf import SYSTEM_IDS, get_conf
from oracle import backward as obw
from oracle import ddp as oddp
from oracle import per as oper
from oracle import rtg as ortg
from oracle import systems as osys

pytestmark = pytest.mark.gpu


def rel_cols(got, want):
    """max |got - want| per column, relative to that column's scale."""
    got, want = np.asarray(got, float), np.asarray(want, float)
    return float((np.abs(got - want) / (np.abs(want).max(axis=0) + 1e-9)).max()) if want.size else 0.0


def setup(system, **over):
    from cacto_b200 import environment as genv
    from cacto_b200.NeuralNetwork import NN
    from cacto_b200.RL import RL_AC
    from cacto_b200.TO import TO_DDP
    conf = get_conf(system, **over)
    env = genv.make_env(conf)
    rl = RL_AC(env, NN(env, conf, 1e-2, seed=0), conf, 0)
    rl.setup_model()
    return conf, env, rl, TO_DDP(env, conf)


def warm_starts(conf, rl, horizon, seed):
    rng = np.random.default_rng(seed)
    X0 = rng.uniform(np.asarray(conf.x_init_min, float), np.asarray(conf.x_init_max, float), (len(horizon), conf.nb_state))
    X0[:, -1] = conf.dt * (conf.NSTEPS - np.asarray(horizon))
    out = rl.rollout_batch(X0, 1, horizon=np.asarray(horizon, dtype=np.int32))
    return X0, out


HORIZONS = {'ur5': [4, 1, 0], 'manipulator': [8, 1, 0, 5]}
MAX_ITER = {'ur5': 4, 'manipulator': 8}


@pytest.mark.parametrize('system', SYSTEM_IDS)
def test_solve_batch_matches_oracle(system):
    conf, env, rl, ddp = setup(system)
    oenv = osys.make_env(conf)
    hz = HORIZONS.get(system, [12, 1, 0, 7])
    max_iter = MAX_ITER.get(system, 12)
    X0, ws = warm_starts(conf, rl, hz, 4)
    res = ddp.solve_batch(X0, ws['states'], ws['controls'], hz, max_iter=max_iter)
    S = res['states'].permute(2, 0, 1).cpu().numpy()
    U = res['controls'].permute(2, 0, 1).cpu().numpy()
    U_in = ws['controls'].permute(2, 0, 1).cpu().numpy()
    cost, status, iters = res['cost'].cpu().numpy(), res['status'].cpu().numpy(), res['iterations'].cpu().numpy()
    hist = res['alpha_index'].cpu().numpy()
    nx = conf.nb_state - 1
    for e, T in enumerate(hz):
        o = oddp.solve(oenv, X0[e, :nx], U_in[e, :T], max_iter=max_iter)
        want_hist = (o['history'] + [oddp.H_NOT_RUN] * 3)[:3]
        assert list(hist[e, :3]) == want_hist, (system, e, hist[e], o['history'])
        assert status[e] == o['status'] and iters[e] == o['iterations'], (system, e)
        assert abs(cost[e] - o['cost']) <= 1e-6 * abs(o['cost']), (system, e, cost[e], o['cost'])
        assert rel_cols(S[e, :T + 1, :nx], o['X']) < 1e-6, (system, e)
        assert rel_cols(U[e, :T], o['U']) < 1e-6, (system, e)
    assert status[hz.index(0)] == oddp.CONVERGED and iters[hz.index(0)] == 0


def test_invariants():
    """Cost non-increasing over iterations; states = an fp64 Env.simulate replay of the controls; x_0 and knots past the horizon
    untouched; a NaN warm start fails alone, leaving every other trajectory's result bit for bit as without it."""
    conf, env, rl, ddp = setup('car', NSTEPS=40)
    hz = [40, 33, 25, 40, 1, 0, 17, 40]
    X0, ws = warm_starts(conf, rl, hz, 7)
    E, nx = len(hz), conf.nb_state - 1
    prev = None
    for n in (0, 1, 2, 3, 5, 8):
        c = ddp.solve_batch(X0, ws['states'], ws['controls'], hz, max_iter=n)['cost'].cpu().numpy()
        if prev is not None:
            assert np.all(c <= prev), (n, c, prev)
        prev = c
    res = ddp.solve_batch(X0, ws['states'], ws['controls'], hz, max_iter=60)
    assert np.all(res['cost'].cpu().numpy() <= res['warm_cost'].cpu().numpy())
    assert (res['status'].cpu().numpy() != ddp.FAILED).all()
    S, U = res['states'], res['controls']
    # replay
    x = torch.as_tensor(X0, device='cuda')
    for t in range(max(hz)):
        x_next = env.simulate_batch(x, U[t].T.contiguous())
        for e in range(E):
            if t < hz[e]:
                want = S[t + 1, :nx, e].cpu().numpy()
                assert np.abs(x_next[e, :nx].cpu().numpy() - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), (t, e)
        x = x_next
    # untouched knots
    same = lambda a, b: bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())
    assert same(S[0], ws['states'][0])
    for e in range(E):
        assert same(S[hz[e] + 1:, :, e], ws['states'][hz[e] + 1:, :, e]) and same(U[hz[e]:, :, e], ws['controls'][hz[e]:, :, e])
        assert same(S[:, nx, e], ws['states'][:, nx, e])                        # the time column
    # NaN warm start
    bad = ws['controls'].clone()
    bad[5, 0, 2] = float('nan')
    res_bad = ddp.solve_batch(X0, ws['states'], bad, hz, max_iter=60)
    assert int(res_bad['status'][2]) == ddp.FAILED and int(res_bad['iterations'][2]) == 0
    keep = [e for e in range(E) if e != 2]
    for k in ('cost', 'status', 'iterations'):
        assert torch.equal(res[k][keep], res_bad[k][keep]), k
    assert same(res['states'][:, :, keep], res_bad['states'][:, :, keep])       # NaN: the rollout's padding past the horizons
    assert same(res['controls'][:, :, keep], res_bad['controls'][:, :, keep])


@pytest.mark.parametrize('system', ['double_integrator', 'manipulator'])
def test_dVdx_is_the_backward_pass_at_the_solution(system):
    from cacto_b200.TO import TO_Casadi
    conf, env, rl, ddp = setup(system)
    hz = [10, 3, 0, 6]
    X0, ws = warm_starts(conf, rl, hz, 11)
    res = ddp.solve_batch(X0, ws['states'], ws['controls'], hz, max_iter=20)
    S = res['states'].permute(2, 0, 1).cpu().numpy()
    U = res['controls'].permute(2, 0, 1).cpu().numpy()
    Vx, off = TO_Casadi(env, conf).backward_pass_batch([S[e, :T + 1] for e, T in enumerate(hz)], [U[e, :T] for e, T in enumerate(hz)])
    assert np.array_equal(off, res['offsets'])
    assert torch.equal(Vx, res['dVdx'])
    for e in range(len(hz)):
        assert np.array_equal(res['dVdx_list'][e], Vx[off[e]:off[e + 1]].cpu().numpy())
        assert np.array_equal(res['TO_states'][e], S[e, :hz[e] + 1])
    # step costs: -reward per knot, summing to the solver's cost
    c = res['step_cost'].cpu().numpy()
    for e in range(len(hz)):
        assert abs(c[off[e]:off[e + 1]].sum() - float(res['cost'][e])) <= 1e-12 * max(1.0, abs(float(res['cost'][e])))


def test_one_episode_of_the_training_loop_with_the_gpu_solve():
    from cacto_b200.replay_buffer import ReplayBuffer
    conf, env, rl, ddp = setup('manipulator', NSTEPS=30, BATCH_SIZE=16, REPLAY_SIZE=2 ** 11)
    conf.UPDATE_LOOPS = np.array([3, 3])
    conf.save_interval = 10 ** 9
    oenv = osys.make_env(conf)
    rng = np.random.default_rng(21)
    n = 6
    X0 = rng.uniform(np.asarray(conf.x_init_min, float), np.asarray(conf.x_init_max, float), (n, conf.nb_state))
    X0[:, -1] = conf.dt * np.round(X0[:, -1] / conf.dt)
    out = rl.rollout_batch(X0, 1)
    assert out['success'].cpu().numpy().all()
    hz = out['horizon'].cpu().numpy()
    res = ddp.solve_batch(X0, out['states'], out['controls'], hz, max_iter=30)
    assert np.all(res['cost'].cpu().numpy() <= res['warm_cost'].cpu().numpy())
    r = rl.rtg_batch(res['TO_states'], res['TO_step_cost'])
    offs = res['offsets']
    cut = lambda t: [t.cpu().numpy()[offs[e]:offs[e + 1]] for e in range(n)]
    buf = ReplayBuffer(conf)
    buf.add(res['TO_states'], cut(r['partial']), cut(r['state_next']), res['dVdx_list'], cut(r['done']), cut(r['term']))
    # the oracle modules on the GPU's own solutions
    U = res['controls'].permute(2, 0, 1).cpu().numpy()
    nx = conf.nb_state - 1
    obuf = oper.ReplayBuffer(conf)
    lists = [[] for _ in range(6)]
    for e in range(n):
        st, ct, T = res['TO_states'][e], U[e, :hz[e]], int(hz[e])
        cost = [oddp.cost_run(oenv, st[t, :nx], ct[t]) for t in range(T)] + [oddp.cost_term(oenv, st[T, :nx])]
        np.testing.assert_allclose(res['TO_step_cost'][e], cost, rtol=1e-12, atol=1e-12)
        dV = obw.backward_pass(oenv, T + 1, st, ct)
        state_arr, partial, total, s_next, done, rwrd, term, ep_ret = ortg.rl_solve(conf, st, cost)
        for l, v in zip(lists, (state_arr, partial, s_next, dV, done, term)):
            l.append(v)
    obuf.add(*lists)
    k = int(sum(hz + 1))
    got, want = buf.storage_mat[:k].cpu().numpy(), obuf.storage_mat[:k]
    ns = conf.nb_state
    rel = lambda a, b: float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))
    assert rel(got[:, :ns], want[:, :ns]) < 1e-9
    assert rel(got[:, ns], want[:, ns]) < 1e-6
    assert rel(got[:, ns + 1:2 * ns + 1], want[:, ns + 1:2 * ns + 1]) < 1e-9
    assert rel(got[:, 2 * ns + 1:3 * ns + 1], want[:, 2 * ns + 1:3 * ns + 1]) < 1e-5
    assert np.array_equal(got[:, 3 * ns + 1:], want[:, 3 * ns + 1:])
    counter = rl.learn_and_update(0, buf, 1)
    assert counter == 3
    for w in rl.critic_model.get_weights() + rl.actor_model.get_weights() + rl.target_critic.get_weights():
        assert np.isfinite(w).all()
