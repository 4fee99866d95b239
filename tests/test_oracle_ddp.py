"""The iLQR oracle (oracle/ddp.py) on the three systems whose optimum is cheap to find another way, at T = 20: its cost never
increases, its adjoint gradient agrees with central differences, the single-shooting gradient vanishes at convergence, and BFGS
on the controls from the same warm start reaches the same cost."""
import numpy as np
import pytest
from scipy.optimize import minimize

from cacto_b200.conf import get_conf
from oracle import ddp as oddp
from oracle import systems as osys

T = 20
SYSTEMS = ['single_integrator', 'double_integrator', 'car']


def warm_start(conf, seed=1):
    rng = np.random.default_rng(seed)
    x0 = rng.uniform(np.asarray(conf.x_init_min[:-1], float), np.asarray(conf.x_init_max[:-1], float))
    U0 = rng.uniform(np.asarray(conf.u_min, float), np.asarray(conf.u_max, float), (T, conf.nb_action)) * 0.1
    return x0, U0


_SOLVED = {}


def solved(system, tol=1e-12):
    if system not in _SOLVED:
        conf = get_conf(system)
        env = osys.make_env(conf)
        x0, U0 = warm_start(conf)
        _SOLVED[system] = conf, env, x0, U0, oddp.solve(env, x0, U0, max_iter=300, tol=tol)
    return _SOLVED[system]


@pytest.mark.parametrize('system', SYSTEMS)
def test_cost_never_increases_and_converges(system):
    conf, env, x0, U0, o = solved(system)
    assert o['status'] == oddp.CONVERGED
    assert np.all(np.diff(o['costs']) <= 0)
    assert o['costs'][-1] < o['costs'][0]
    assert any(h >= 0 for h in o['history'])
    # the committed iterate is the rollout of its controls
    J, X, _ = oddp.rollout(env, x0, o['U'])
    assert J == o['cost'] and np.array_equal(X, o['X'])


@pytest.mark.parametrize('system', SYSTEMS)
def test_adjoint_gradient_matches_central_differences(system):
    conf, env, x0, U0, _ = solved(system)
    g = oddp.gradient(env, oddp.rollout(env, x0, U0)[1], U0)
    rng = np.random.default_rng(3)
    for t, a in [(0, 0), (T // 2, 1), (T - 1, rng.integers(conf.nb_action))]:
        h = 1e-6 * max(1.0, abs(U0[t, a]))
        Up, Um = U0.copy(), U0.copy()
        Up[t, a] += h
        Um[t, a] -= h
        fd = (oddp.total_cost(env, x0, Up) - oddp.total_cost(env, x0, Um)) / (2 * h)
        assert abs(fd - g[t, a]) <= 1e-6 * np.abs(g).max(), (t, a, fd, g[t, a])


@pytest.mark.parametrize('system', SYSTEMS)
def test_gradient_vanishes_at_convergence(system):
    """dJ/dU relative to the cost and the control range: the change of J per full-scale control move."""
    conf, env, x0, U0, o = solved(system)
    g = oddp.gradient(env, o['X'], o['U'])
    assert np.abs(g).max() * np.max(conf.u_max) <= 1e-6 * abs(o['cost'])


@pytest.mark.parametrize('system', SYSTEMS)
def test_bfgs_from_the_same_warm_start_reaches_the_same_cost(system):
    conf, env, x0, U0, o = solved(system)

    def fg(v):
        U = v.reshape(U0.shape)
        J, X, _ = oddp.rollout(env, x0, U)
        return J, oddp.gradient(env, X, U).ravel()
    r = minimize(fg, U0.ravel(), jac=True, method='BFGS', options=dict(gtol=1e-10, maxiter=2000))
    assert abs(r.fun - o['cost']) <= 1e-6 * abs(o['cost']), (r.fun, o['cost'])


def test_tolerance_trades_iterations_for_accuracy():
    conf, env, x0, U0, tight = solved('car')
    loose = oddp.solve(env, x0, U0, max_iter=300, tol=1e-8)
    assert loose['status'] == oddp.CONVERGED and loose['iterations'] <= tight['iterations']
    assert tight['cost'] <= loose['cost'] <= tight['cost'] + 1e-6 * abs(tight['cost'])


def test_non_finite_warm_start_fails_and_empty_horizon_converges():
    conf = get_conf('single_integrator')
    env = osys.make_env(conf)
    x0, U0 = warm_start(conf)
    U0[3, 0] = np.nan
    o = oddp.solve(env, x0, U0)
    assert o['status'] == oddp.FAILED and o['iterations'] == 0
    o = oddp.solve(env, x0, np.zeros((0, conf.nb_action)))
    assert o['status'] == oddp.CONVERGED and o['cost'] == oddp.cost_term(env, x0)
