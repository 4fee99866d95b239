"""Trained networks for the accuracy tests: the reference's own trained double-integrator nets (tests/golden/h5_di_try6_final.npz,
make_golden.py) and, for every system, deterministic "trained-scale" nets with the magnitudes of those (non-zero biases, per-layer
max|W| of the trained net, heavy-tailed kernels), plus batches of states such a policy visits.

At construction (NeuralNetwork.py create_*) every actor bias is 0 and all kernel entries have a similar size; a kernel that
dropped or misindexed a bias, or whose max-based fp16 scaling misbehaved when a few entries dominate, would not show there.
A plain helper module (not a fixture): test_trained_nets.py checks what it delivers, test_gpu_trained_nets.py uses it."""
import functools
import os

import numpy as np
import torch

from oracle import nn as onn
from oracle import rtg as ortg
from oracle import systems as osys

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')

# Magnitudes of the trained DI networks (h5_di_try6_final.npz): per layer max|W| and the standard deviation of the bias.
ACTOR_WMAX = (0.65, 1.11, 1.84)
ACTOR_BSIG = (0.088, 0.096, 0.097)
CRITIC_WMAX = (1.77, 0.61, 0.86, 0.83)          # hidden layers; the head below
CRITIC_BSIG = (0.28, 0.22, 0.20, 0.25)
HEAD_W, HEAD_B = 6.0, 4.3
TAIL_FRAC = 0.03                                # share of kernel entries at 2-3x the bulk: they set max|W|
TARGET_PERTURB = 1e-2                           # target critic = critic * (1 + 1e-2 N(0, 1))


def di_trained():
    """(actor, critic, target_critic) weight lists of the trained DI networks, exactly as stored."""
    g = np.load(os.path.join(GOLDEN, 'h5_di_try6_final.npz'))
    return ([g[f'actor_{i}'] for i in range(6)], [g[f'critic_{i}'] for i in range(10)], [g[f'target_critic_{i}'] for i in range(10)])


def _kernel(rng, i, o, wmax):
    """Uniform bulk with a heavy tail: TAIL_FRAC of the entries at 2-3x the bulk's range; scaled so that max|W| == wmax."""
    w = rng.uniform(-1.0, 1.0, (i, o))
    tail = rng.uniform(size=(i, o)) < TAIL_FRAC
    w[tail] = np.sign(w[tail]) * rng.uniform(2.0, 3.0, int(tail.sum()))
    k = np.unravel_index(int(rng.integers(w.size)), w.shape)       # at least one outlier, whatever the shape
    w[k] = 3.0
    return (w * (wmax / np.abs(w).max())).astype(np.float32)


def _bias(rng, o, sig):
    b = rng.normal(0.0, sig, o)
    b[np.abs(b) < 1e-3 * sig] = sig                                 # every entry non-zero
    return b.astype(np.float32)


def _critic(rng, dims):
    """dims = [ns, h1, h2, h3, h4, 1]: hidden layers at the DI critic's per-layer magnitudes, head of the DI head's size."""
    p = []
    for l, (i, o) in enumerate(zip(dims[:-2], dims[1:-1])):
        p += [_kernel(rng, i, o, CRITIC_WMAX[l]), _bias(rng, o, CRITIC_BSIG[l])]
    p += [_kernel(rng, dims[-2], 1, HEAD_W), np.array([HEAD_B], np.float32)]
    return p


LEAKY_PAIR = 1.3                 # leaky(z) - leaky(-z) = 1.3 z for LeakyReLU(0.3): a unit pair passes z through linearly
FEEDBACK_KMAX = 4.0              # largest feedback gain, action per unit of normalised state
RANDOM_OUT = 0.25                # the random units' share of max|W3|: small enough that the embedded feedback keeps the loop bounded


def _feedback_gain(conf):
    """LQR gain K (u = -K (xn - xn0), xn the normalised state without time) of the fp64 oracle dynamics linearised at the centre of
    the x_init box with u = 0.  A 0.999 discount makes the DARE solvable where a mode is not controllable (the car's heading and
    lateral position at v = 0)."""
    import scipy.linalg
    env = osys.make_env(conf)
    nx, na = conf.nb_state - 1, conf.nb_action
    norm = np.asarray(conf.state_norm_arr, float)[:nx]
    x0 = 0.5 * (np.asarray(conf.x_init_min, float) + np.asarray(conf.x_init_max, float))
    x0[-1] = 0.0
    f = lambda x, u: env.simulate(x, u)[:nx] / norm
    A, B, h = np.zeros((nx, nx)), np.zeros((nx, na)), 1e-6
    for i in range(nx):
        d = np.zeros(nx + 1); d[i] = h * norm[i]
        A[:, i] = (f(x0 + d, np.zeros(na)) - f(x0 - d, np.zeros(na))) / (2 * h)
    for j in range(na):
        d = np.zeros(na); d[j] = h
        B[:, j] = (f(x0, d) - f(x0, -d)) / (2 * h)
    A = 0.999 * A

    def gain(r):
        P = scipy.linalg.solve_discrete_are(A, B, np.eye(nx), r * np.eye(na))
        return np.linalg.solve(r * np.eye(na) + B.T @ P @ B, B.T @ P @ A)
    lo, hi = -8.0, 4.0                        # log10 of the control weight: max|K| = FEEDBACK_KMAX (actions of a trained size)
    for _ in range(40):
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if np.abs(gain(10 ** mid)).max() > FEEDBACK_KMAX else (lo, mid)
    return gain(10 ** hi), x0[:nx] / norm


def _actor(rng, conf, nh):
    """A trained-scale actor (the recipe above) that is also a stabilising policy, as a trained one is: it computes
    u = -K (xn - xn0) + r(x) exactly, the LQR feedback through LeakyReLU unit pairs of both hidden layers and r the recipe's random
    units with their output weights at RANDOM_OUT of max|W3|."""
    ns, na, nx = conf.nb_state, conf.nb_action, conf.nb_state - 1
    K, xn0 = _feedback_gain(conf)
    W1, b1 = _kernel(rng, ns, nh[0], ACTOR_WMAX[0]), _bias(rng, nh[0], ACTOR_BSIG[0])
    W2, b2 = _kernel(rng, nh[0], nh[1], ACTOR_WMAX[1]), _bias(rng, nh[1], ACTOR_BSIG[1])
    W3, b3 = _kernel(rng, nh[1], na, ACTOR_WMAX[2]), _bias(rng, na, ACTOR_BSIG[2])
    W3 *= RANDOM_OUT
    a = ACTOR_WMAX[0]
    copies = int(np.ceil(np.abs(K).max() / (LEAKY_PAIR ** 2 * a * ACTOR_WMAX[1] * ACTOR_WMAX[2])))
    c = np.abs(K).max() / (LEAKY_PAIR ** 2 * a * copies * ACTOR_WMAX[2])        # <= max|W2|: the pairs' layer-3 weights reach max|W3|
    n = 2 * nx * copies
    assert n <= min(nh), (n, nh)
    W2[:, :n] = 0.0                                                             # the pass-through columns see only their pair
    offset = np.zeros(na)
    for k in range(copies):
        for i in range(nx):
            p = 2 * (k * nx + i)
            W1[:, p:p + 2] = 0.0
            W1[i, p], W1[i, p + 1] = a, -a
            b1[p + 1] = -b1[p]                                                  # h1[p] - h1[p+1] = 1.3 (a xn_i + b1[p])
            W2[p, p], W2[p + 1, p], W2[p, p + 1], W2[p + 1, p + 1] = c, -c, -c, c
            b2[p + 1] = -b2[p]                                                  # h2[p] - h2[p+1] = 1.3 (1.3 c (a xn_i + b1[p]) + b2[p])
            g = -K[:, i] / (LEAKY_PAIR ** 2 * a * c * copies)
            W3[p], W3[p + 1] = g, -g
            offset += g * LEAKY_PAIR * (LEAKY_PAIR * c * b1[p] + b2[p])
    b3 = b3 - offset + K @ xn0                                                  # the pairs' constant terms and the set point
    return [W1.astype(np.float32), b1, W2.astype(np.float32), b2, W3.astype(np.float32), b3.astype(np.float32)]


def trained_scale(system, critic_type='sine', seed=0, nh=(256, 256)):
    """(conf, actor, critic, target) weight lists for ``system``, deterministic in ``seed``: the recipe above on the init shapes
    of the actor and of ``critic_type``'s critic ('sine', 'elu', 'sine-elu', 'relu'); the actor is a stabilising policy (_actor)."""
    from cacto_b200.conf import get_conf
    conf = get_conf(system, critic_type=critic_type, NH1=nh[0], NH2=nh[1])
    rng = np.random.default_rng([seed, sum(map(ord, system)), sum(map(ord, critic_type))])
    actor = _actor(rng, conf, nh)
    critic = _critic(rng, [conf.nb_state] + list(onn.critic_spec(conf)[0]) + [1])
    target = [(c * (1 + TARGET_PERTURB * rng.standard_normal(c.shape))).astype(np.float32) for c in critic]
    return conf, actor, critic, target


def rollouts64(conf, actor, X0, steps=None):
    """fp64 oracle rollouts (RL.py create_TO_init with the fp64 actor): states [B, T+1, ns] (NaN past each horizon), controls."""
    env = osys.make_env(conf)
    X0 = np.asarray(X0, float)
    hz = np.array([ortg.horizon(conf, x[-1]) for x in X0])
    T = int(hz.max() if steps is None else min(steps, hz.max()))
    S = np.full((len(X0), T + 1, conf.nb_state), np.nan)
    U = np.full((len(X0), T, conf.nb_action), np.nan)
    S[:, 0] = X0
    for t in range(T):
        live = np.flatnonzero(hz > t)
        U[live, t] = actor64(actor, conf, S[live, t])
        for b in live:
            S[b, t + 1] = env.simulate(S[b, t], U[b, t])
    return S, U


def h1_of(actor, conf, s):
    """fp64 first hidden layer (after LeakyReLU) of the actor at states s."""
    p = onn.to_torch(actor, torch.float64)
    x = onn.normalize(torch.as_tensor(np.asarray(s, np.float64)), conf.state_norm_arr)
    return torch.nn.functional.leaky_relu(x @ p[0] + p[1], 0.3).numpy()


def scaled(weights, h1_target, conf, s):
    """The actor with W1, b1 multiplied and W2 divided by one factor, chosen so that the fp64 max|h1| over the states s equals
    h1_target.  LeakyReLU is positively homogeneous, so the actions are unchanged (up to the fp32 rounding of the weights)."""
    k = h1_target / float(np.abs(h1_of(weights, conf, s)).max())
    w = [x.copy() for x in weights]
    w[0], w[1], w[2] = (w[0] * k).astype(np.float32), (w[1] * k).astype(np.float32), (w[2] / k).astype(np.float32)
    return w


def actor64(actor, conf, s):
    with torch.no_grad():
        return onn.actor_forward(onn.to_torch(actor, torch.float64), torch.as_tensor(np.asarray(s, np.float64)), conf).numpy()


def box(conf, B, rng):
    """States uniform in the x_init box; time on the dt grid, the first and last rows at t = 0 and at the last step."""
    lo, hi = np.asarray(conf.x_init_min, float), np.asarray(conf.x_init_max, float)
    x = rng.uniform(lo, hi, (B, conf.nb_state))
    x[:, -1] = conf.dt * rng.integers(0, conf.NSTEPS, B)
    x[0, -1], x[-1, -1] = 0.0, (conf.NSTEPS - 1) * conf.dt
    return x


# distinct visited states per system: the oracle's per-sample dynamics cost up to ~10 ms (UR5), so the pool is small and cached
_POOL_TRAJ, _POOL_STEPS = 16, 16


@functools.lru_cache(maxsize=None)
def _visited(system, seed):
    conf, actor = trained_scale(system, seed=seed)[:2]
    env = osys.make_env(conf)
    rng = np.random.default_rng([seed, 7])
    out = []
    for x0 in box(conf, _POOL_TRAJ, rng):
        x = x0
        for _ in range(min(_POOL_STEPS, ortg.horizon(conf, x[-1]))):
            x = env.simulate(x, actor64(actor, conf, x[None])[0])
            if not np.isfinite(x).all():
                break
            x[-1] = conf.dt * round(x[-1] / conf.dt)
            out.append(x)
    return np.array(out)


def states(conf, B, seed=0):
    """[B, ns] float32: half from the x_init box, half from fp64 oracle rollouts of the trained-scale actor of seed ``seed``
    (these may leave the box), jittered by 1e-3 of the state norm so that resampled pool entries are distinct."""
    rng = np.random.default_rng([seed, B])
    nb = B - B // 2
    s = np.empty((B, conf.nb_state))
    s[:nb] = box(conf, nb, rng)
    pool = _visited(conf.system_id, seed)
    v = pool[rng.integers(0, len(pool), B // 2)]
    v[:, :-1] += 1e-3 * np.asarray(conf.state_norm_arr[:-1], float) * rng.standard_normal((B // 2, conf.nb_state - 1))
    s[nb:] = v
    return s.astype(np.float32)


def update_batch(conf, B, seed=0):
    """(state, partial_rtg, state_next, dVdx, done, term, weights) for the critic / actor gradients at trained-network
    magnitudes (rtg of the size the DI critic predicts, dV/dx from N(0, 1))."""
    rng = np.random.default_rng([seed, B, 3])
    s = states(conf, B, seed)
    sn = states(conf, B, seed + 1)
    pr = rng.uniform(-20, 0, (B, 1)).astype(np.float32)
    dv = rng.normal(size=(B, conf.nb_state)).astype(np.float32)
    dv[:, -1] = 0
    d = (rng.uniform(size=(B, 1)) < 0.5).astype(np.float32)
    term = (rng.uniform(size=(B, 1)) < 0.2).astype(np.float64)
    w = rng.uniform(0.2, 1.5, (B, 1)).astype(np.float32)
    return s, pr, sn, dv, d, term, w
