"""CPU restatement of the batched iLQR TO solver (kernel K7, csrc/ddp.cu) -- ORACLE, test infrastructure only.

The problem (include/cacto_b200.h states it once more): from x_0 (no time column) minimise over U = (u_0 .. u_{T-1})

    J(U) = sum_{k<T} c_run(x_k, u_k) + c_term(x_T),   x_{k+1} = Env.simulate(x_k, u_k),

with c = -reward (running / terminal weights) and the bounded control cost a^2 + w_b (a/u_max)^10 for every system, UR5
included (quirk Q8): ``oracle.backward.reward_generic``, whose derivatives K6 evaluates.  No hard bounds (quirk Q11).
iLQR is a local method: nothing here claims equality with ipopt's solutions.

One iteration: derivatives at the iterate (``oracle.backward``), the backward recursion on the cost with a Cholesky factor of
Q_uu + mu I (failure: mu grows, no step), gains k = -Quu~^-1 Q_u, K = -Quu~^-1 Q_ux, V_x = Q_x + K'Q_uu k + K'Q_u + Q_ux'k,
V_xx = sym(Q_xx + K'Q_uu K + K'Q_ux + Q_ux'K), expected change dV(a) = a dV1 + a^2/2 dV2; closed-loop probes at a = 2^-j,
j < N_ALPHA; the largest a with J - J(a) >= C1 (-dV(a)) is taken.  Constants, statuses and history codes mirror the header's.
"""
import numpy as np

from . import backward as obw

N_ALPHA = 8
C1 = 1e-4
MU_INIT = 1e-6
MU_MIN = 1e-9
MU_MAX = 1e10
MU_FACTOR = 10.0
HISTORY = 8
RUNNING, CONVERGED, FAILED = 0, 1, 2
H_BACKWARD_FAILED, H_NO_STEP, H_CONVERGED, H_NOT_RUN = -1, -2, -3, -4


def step(env, x, u):
    return np.asarray(env.simulate(np.append(x, 0.0), u), dtype=float)[:-1]


def cost_run(env, x, u):
    return -obw.reward_generic(env, env.conf.cost_weights_running, list(x), list(u))


def cost_term(env, x):
    return -obw.reward_generic(env, env.conf.cost_weights_terminal, list(x))


def rollout(env, x0, U_bar, X_bar=None, k=None, K=None, alpha=0.0):
    """Open loop (k is None) or closed loop u_t = u_bar_t + alpha k_t + K_t (x_t - x_bar_t).  Returns (J, X[T+1, nx], U[T, na])."""
    T = len(U_bar)
    X = np.empty((T + 1, len(x0)))
    U = np.array(U_bar, dtype=float)                                     # [T, na], a copy
    X[0] = x0
    J = 0.0
    with np.errstate(all='ignore'):
        for t in range(T):
            if k is not None:
                U[t] = U_bar[t] + alpha * k[t] + K[t] @ (X[t] - X_bar[t])
            J += cost_run(env, X[t], U[t])
            X[t + 1] = step(env, X[t], U[t])
        J += cost_term(env, X[T])
    return J, X, U


def knot_derivatives(env, x, u=None):
    """Cost derivatives (l_x, l_xx[, l_u, l_uu, A, B]) at one knot: the reward's, negated; A, B = Env.augmented_derivative."""
    c = env.conf
    if u is None:
        gx, Hx = obw.reward_x_derivatives(env, c.cost_weights_terminal, x)
        return -gx, -Hx
    gx, Hx = obw.reward_x_derivatives(env, c.cost_weights_running, x)
    gu, Hu = obw.reward_u_derivatives(env, c.cost_weights_running, u)
    A, B = env.augmented_derivative(np.append(x, 0.0), u)
    return -gx, -Hx, -gu, -Hu, np.asarray(A, dtype=float), np.asarray(B, dtype=float)


def backward(env, X, U, mu):
    """Returns (ok, k[T, na], K[T, na, nx], dV1, dV2)."""
    T, na, nx = len(U), U.shape[1], X.shape[1]
    lx, lxx = knot_derivatives(env, X[T])
    Vx, Vxx = lx, lxx
    k, K = np.zeros((T, na)), np.zeros((T, na, nx))
    dv1 = dv2 = 0.0
    for t in range(T - 1, -1, -1):
        lx, lxx, lu, luu, A, B = knot_derivatives(env, X[t], U[t])
        Qx = lx + A.T @ Vx
        Qu = lu + B.T @ Vx
        Qxx = lxx + A.T @ Vxx @ A
        Quu = luu + B.T @ Vxx @ B
        Qux = B.T @ Vxx @ A                                              # l_ux = 0: the cost is separable
        M = 0.5 * (Quu + Quu.T) + mu * np.identity(na)
        with np.errstate(all='ignore'):
            try:
                L = np.linalg.cholesky(M)
            except np.linalg.LinAlgError:
                return False, k, K, dv1, dv2
        if not np.all(np.isfinite(L)) or not np.all(np.diag(L) > 0):
            return False, k, K, dv1, dv2
        sol = np.linalg.solve(L.T, np.linalg.solve(L, -np.column_stack([Qu, Qux])))
        k[t], K[t] = sol[:, 0], sol[:, 1:]
        dv1 += k[t] @ Qu
        dv2 += k[t] @ (Quu @ k[t])
        Vx = Qx + K[t].T @ (Quu @ k[t]) + K[t].T @ Qu + Qux.T @ k[t]
        V = Qxx + K[t].T @ (Quu @ K[t]) + K[t].T @ Qux + Qux.T @ K[t]
        Vxx = 0.5 * (V + V.T)
    return True, k, K, dv1, dv2


def solve(env, x0, U0, max_iter=100, tol=1e-8):
    """iLQR from the warm start U0[T, na] at x0[nx].  Returns a dict: X, U, cost, status, iterations, history (accepted alpha index
    per iteration, or an H_* code), costs (J after every iteration, the warm start's first)."""
    x0 = np.asarray(x0, dtype=float)
    U0 = np.asarray(U0, dtype=float).reshape(len(U0), -1) if len(U0) else np.zeros((0, env.conf.nb_action))
    J, X, U = rollout(env, x0, U0)
    out = dict(history=[], costs=[J])
    status = FAILED if not np.isfinite(J) else (CONVERGED if len(U) == 0 else RUNNING)
    mu, it = MU_INIT, 0
    while status == RUNNING and it < max_iter:
        it += 1
        ok, k, K, dv1, dv2 = backward(env, X, U, mu)
        if not ok:
            outcome = H_BACKWARD_FAILED
        elif abs(dv1 + 0.5 * dv2) < tol * abs(J):
            outcome = H_CONVERGED
        else:
            outcome = H_NO_STEP
            for j in range(N_ALPHA):
                a = 2.0 ** -j
                Jp = rollout(env, x0, U, X, k, K, a)[0]
                expected = -(a * dv1 + 0.5 * a * a * dv2)
                if np.isfinite(Jp) and expected > 0 and J - Jp >= C1 * expected:
                    outcome = j
                    break
        out['history'].append(outcome)
        if outcome >= 0:
            Jn, X, U = rollout(env, x0, U, X, k, K, 2.0 ** -outcome)
            mu = max(mu / MU_FACTOR, MU_MIN)
            if J - Jn < tol * abs(J):
                status = CONVERGED
            J = Jn
        elif outcome == H_CONVERGED:
            status = CONVERGED
        else:
            mu *= MU_FACTOR
            if mu > MU_MAX:
                status = FAILED
        out['costs'].append(J)
    out.update(X=X, U=U, cost=J, status=status, iterations=it)
    return out


def _cost_x_gradient(env, weights, x):
    """First derivatives of x -> -reward_generic (one hyper-dual evaluation per coordinate, no Hessian)."""
    n = len(x)
    g = np.empty(n)
    for i in range(n):
        xs = [obw.HD(x[j], 1.0 if j == i else 0.0) for j in range(n)]
        g[i] = -obw.HD.lift(obw.reward_generic(env, weights, xs)).a
    return g


def gradient(env, X, U):
    """Single-shooting gradient dJ/dU[T, na] along the rollout (X, U), by the adjoint recursion."""
    c = env.conf
    T = len(U)
    lam = _cost_x_gradient(env, c.cost_weights_terminal, X[T])
    g = np.zeros_like(np.asarray(U, dtype=float))
    for t in range(T - 1, -1, -1):
        A, B = env.augmented_derivative(np.append(X[t], 0.0), U[t])
        lu = -obw.reward_u_derivatives(env, c.cost_weights_running, U[t])[0]
        g[t] = lu + np.asarray(B).T @ lam
        lam = _cost_x_gradient(env, c.cost_weights_running, X[t]) + np.asarray(A).T @ lam
    return g


def total_cost(env, x0, U):
    return rollout(env, np.asarray(x0, dtype=float), np.asarray(U, dtype=float).reshape(len(U), -1))[0]
