"""CPU restatement of NeuralNetwork.py / RL.py's update (torch-CPU autograd) -- ORACLE, test only.

PARITY UNPINNED: TensorFlow 2.11 / Keras 2.11 / tf_siren 0.0.5 are not installable in the
build container and the reference ships no loss/gradient vectors.  What this file follows:

* network shapes and initialisers: NeuralNetwork.py:51-63 (actor), :95-108 (critic 'sine'),
  confirmed by the archived .h5 weight files (tests/golden/h5_*.npz);
* ``normalize_tensor``: utils.py:17-24;
* Keras semantics (published behaviour): Dense = x @ kernel(in, out) + bias; LeakyReLU
  alpha = 0.3; MeanSquaredError(sample_weight) = sum_i w_i * mean_j(d_ij^2) / B;
  tf.maximum passes the gradient to x when x >= y;
* TF-2.11 Adam (new-style optimizer): eps = 1e-7 added outside the bias correction.

Parameters are lists of arrays [W1, b1, W2, b2, ...] with Keras' (in, out) kernel layout.
"""
import math

import numpy as np
import torch

CRITIC_HIDDEN = (64, 64, 128, 128)


# ----------------------------------------------------------------------------- initialisers
def init_actor(ns, na, nh1=256, nh2=256, seed=0):
    """Dense glorot-uniform kernels, zero biases (Keras defaults)."""
    rng = np.random.default_rng(seed)
    dims = [ns, nh1, nh2, na]
    p = []
    for i, o in zip(dims[:-1], dims[1:]):
        lim = math.sqrt(6.0 / (i + o))
        p += [rng.uniform(-lim, lim, (i, o)).astype(np.float32), np.zeros(o, np.float32)]
    return p


def init_critic_sine(ns, seed=0):
    """SIREN layers: kernel U(+-sqrt(6/fan_in)) (w0 = 1), bias he_uniform U(+-sqrt(6/units));
    final Dense(1) glorot-uniform, zero bias."""
    rng = np.random.default_rng(seed)
    dims = [ns] + list(CRITIC_HIDDEN)
    p = []
    for i, o in zip(dims[:-1], dims[1:]):
        lk, lb = math.sqrt(6.0 / i), math.sqrt(6.0 / o)
        p += [rng.uniform(-lk, lk, (i, o)).astype(np.float32), rng.uniform(-lb, lb, o).astype(np.float32)]
    lim = math.sqrt(6.0 / (dims[-1] + 1))
    p += [rng.uniform(-lim, lim, (dims[-1], 1)).astype(np.float32), np.zeros(1, np.float32)]
    return p


def to_torch(params, dtype=torch.float32, requires_grad=False):
    return [torch.tensor(np.asarray(a), dtype=dtype, requires_grad=requires_grad) for a in params]


# ----------------------------------------------------------------------------- forward passes
def normalize(x, norm):
    """utils.py:17-24: x/norm for the state part, 2 t/T - 1 for the time (last) column."""
    norm = torch.as_tensor(np.asarray(norm, dtype=np.float64), dtype=x.dtype)
    xn = x / norm
    return torch.cat([xn[:, :-1], xn[:, -1:] * 2 - 1], dim=1)


def actor_forward(p, s, conf):
    x = normalize(s, conf.state_norm_arr) if conf.NORMALIZE_INPUTS else s
    h = torch.nn.functional.leaky_relu(x @ p[0] + p[1], 0.3)
    h = torch.nn.functional.leaky_relu(h @ p[2] + p[3], 0.3)
    return h @ p[4] + p[5]


def critic_spec(conf):
    """(hidden widths, activation per hidden layer, is-SIREN per hidden layer) of conf.critic_type:
    NeuralNetwork.py:95-108 'sine', :65-78 'elu', :80-93 'sine-elu', :110-128 'relu' (LeakyReLU() = alpha 0.3)."""
    t = getattr(conf, 'critic_type', 'sine')
    if t == 'sine':
        return CRITIC_HIDDEN, ('sin',) * 4, (True,) * 4
    if t == 'elu':
        return (16, 32, 256, 256), ('elu',) * 4, (False,) * 4
    if t == 'sine-elu':
        return (64, 64, 128, 128), ('sin', 'elu', 'sin', 'elu'), (True, False, True, False)
    return (16, 32, conf.NH1, conf.NH2), ('leaky',) * 4, (False,) * 4


_ACT = {'sin': torch.sin, 'elu': torch.nn.functional.elu, 'leaky': lambda z: torch.nn.functional.leaky_relu(z, 0.3)}


def critic_forward(p, s, conf):
    x = normalize(s, conf.state_norm_arr) if conf.NORMALIZE_INPUTS else s
    acts = critic_spec(conf)[1]
    h = x
    for l in range(4):
        h = _ACT[acts[l]](h @ p[2 * l] + p[2 * l + 1])
    return h @ p[8] + p[9]


def slog(x):
    """NeuralNetwork.py:140-148 (custom_logarithm)."""
    pos = torch.log(torch.clamp(x, min=1e-7) + 1)
    neg = -torch.log(torch.clamp(-x, min=1e-7) + 1)
    return torch.where(x > 0, pos, neg)


def _wmse(y_true, y_pred, w):
    per = ((y_pred - y_true) ** 2).mean(dim=-1)
    return (per * w.reshape(-1)).sum() / per.shape[0]


# ----------------------------------------------------------------------------- gradients
def critic_grad(critic, target, conf, w_S, state, state_next, partial_rtg, dVdx, d, weights, dtype=torch.float32):
    """NeuralNetwork.py:150-178.  Returns (grads, rtg, V, V_target(state), loss) as NumPy."""
    cp = to_torch(critic, dtype, True)
    tp = to_torch(target, dtype)
    t = lambda a: torch.tensor(np.asarray(a), dtype=dtype)
    s, sn, pr, dv, dd, w = t(state), t(state_next), t(partial_rtg), t(dVdx), t(d), t(weights)
    if conf.MC:
        rtg = pr
    else:
        with torch.no_grad():
            rtg = pr + (1 - dd) * critic_forward(tp, sn, conf)
    if w_S != 0:
        s.requires_grad_(True)
        V = critic_forward(cp, s, conf)
        dVds, = torch.autograd.grad(V.sum(), s, create_graph=True)
        loss_v = _wmse(rtg, V, w)
        loss_d = _wmse(slog(dv[:, :-1]), slog(dVds[:, :-1]), w)
        loss = loss_d + w_S * loss_v
    else:
        V = critic_forward(cp, s, conf)
        loss = _wmse(rtg, V, w)
    grads = torch.autograd.grad(loss, cp)
    with torch.no_grad():
        Vt = critic_forward(tp, t(state), conf)
    return ([g.numpy() for g in grads], rtg.numpy(), V.detach().numpy(), Vt.numpy(), float(loss.detach()))


def actor_grad(actor, critic, conf, env, state, term, dtype=torch.float32):
    """NeuralNetwork.py:180-232.  ``env`` is an oracle.systems environment.
    Returns (grads, actions, state_next, dQ_da) as NumPy."""
    ap = to_torch(actor, dtype, True)
    cp = to_torch(critic, dtype)
    s = torch.tensor(np.asarray(state), dtype=dtype)
    B = s.shape[0]
    with torch.no_grad():
        a0 = actor_forward(ap, s, conf)
    s_np, a_np = s.numpy(), a0.numpy()
    s_next = torch.tensor(env.simulate_batch(s_np, a_np), dtype=dtype, requires_grad=True)
    Fu = torch.tensor(env.derivative_batch(s_np, a_np), dtype=dtype)
    Vn = critic_forward(cp, s_next, conf)
    dV, = torch.autograd.grad(Vn.sum(), s_next)

    term = np.asarray(term, dtype=np.float64).reshape(-1, 1)
    wt = np.reshape(conf.cost_weights_terminal, [1, -1])
    wr = np.reshape(conf.cost_weights_running, [1, -1])
    wts = term.dot(wt) + (1 - term).dot(wr)
    a1 = a0.clone().requires_grad_(True)
    u_max = torch.tensor(np.asarray(conf.u_max, dtype=np.float64), dtype=dtype)
    u_cost = (a1 ** 2 + conf.w_b * (a1 / u_max) ** 10).sum(dim=1)
    scale = float(conf.cost_funct_param[1])
    r = scale * (-torch.tensor(wts[:, 6], dtype=dtype) * u_cost)        # state part is constant w.r.t. a
    dr_da, = torch.autograd.grad(r.sum(), a1)
    dQ_da = torch.matmul(dV.reshape(B, 1, -1), Fu).reshape(B, -1) + dr_da
    a = actor_forward(ap, s, conf)
    mean_Qneg = (-(dQ_da.detach()) * a).sum(dim=1).mean()
    grads = torch.autograd.grad(mean_Qneg, ap)
    return ([g.numpy() for g in grads], a0.numpy(), s_next.detach().numpy(), dQ_da.detach().numpy())


# ----------------------------------------------------------------------------- optimiser
def piecewise_lr(step, boundaries, values):
    """PiecewiseConstantDecay: values[#{b < step}] (RL.py:82-85)."""
    return values[sum(1 for b in boundaries if b < step)]


class Adam:
    """tf.keras.optimizers.Adam of TF 2.11 (new-style optimizer), float32 arithmetic."""

    def __init__(self, params, lr, beta1=0.9, beta2=0.999, eps=1e-7):
        self.lr, self.b1, self.b2, self.eps = lr, beta1, beta2, eps
        self.m = [np.zeros_like(p) for p in params]
        self.v = [np.zeros_like(p) for p in params]
        self.iterations = 0

    def current_lr(self):
        return self.lr(self.iterations) if callable(self.lr) else self.lr

    def apply_gradients(self, params, grads):
        f = np.float32
        lr = f(self.current_lr())
        t = f(self.iterations + 1)
        alpha = lr * np.sqrt(f(1) - np.power(f(self.b2), t)) / (f(1) - np.power(f(self.b1), t))
        for i, (p, g) in enumerate(zip(params, grads)):
            g = g.astype(f)
            self.m[i] += (g - self.m[i]) * f(1 - self.b1)
            self.v[i] += (g * g - self.v[i]) * f(1 - self.b2)
            p -= (self.m[i] * alpha) / (np.sqrt(self.v[i]) + f(self.eps))
        self.iterations += 1


def polyak(target, source, tau):
    """RL.py:113-118."""
    f = np.float32
    for a, b in zip(target, source):
        a[...] = b * f(tau) + a * f(1 - tau)


def update(critic, target, actor, opt_c, opt_a, conf, w_S, env, batch, dtype=torch.float32):
    """One RL_AC.update + update_target (RL.py:101-111,134-135).  ``batch`` =
    (state, partial_rtg, state_next, dVdx, d, term, weights).  In-place on the parameter lists.  ``dtype`` is the precision of
    the gradients (as in critic_grad / actor_grad); Adam and Polyak stay in float32 as in the reference."""
    state, partial_rtg, state_next, dVdx, d, term, weights = batch
    cg, rtg, V, Vt, loss = critic_grad(critic, target, conf, w_S, state, state_next, partial_rtg, dVdx, d, weights, dtype=dtype)
    opt_c.apply_gradients(critic, cg)
    ag, actions, s_next, dQ = actor_grad(actor, critic, conf, env, state, term, dtype=dtype)
    opt_a.apply_gradients(actor, ag)
    if not conf.MC:
        polyak(target, critic, conf.UPDATE_RATE)
    return dict(critic_grad=cg, actor_grad=ag, rtg=rtg, V=V, V_target=Vt, loss=loss, actions=actions,
                state_next=s_next, dQ_da=dQ)
