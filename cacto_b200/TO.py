"""Host mirror of the GPU-resident part of the reference's TO.py: ``TO_Casadi.backward_pass`` (TO.py:119-202), and a GPU TO solver.

The CasADi / ipopt solves (``TO_System_Solve``, ``TO_Solve``) stay on the host pool of the reference (north_star: out of
scope here); what moves to the GPU is the per-knot Python loop that turns a TO solution into ``dVdx`` -- kernel K6
(``cacto_backward_pass``, csrc/backward.cu).  ``backward_pass`` keeps the reference's signature and return value;
``backward_pass_batch`` processes all TO solutions of an episode batch in one launch pair.

``TO_DDP`` is an opt-in alternative to the ipopt solve: batched iLQR on the GPU (kernel K7, csrc/ddp.cu) for the same optimal
control problem, warm-started from ``RL_AC.rollout_batch`` (include/cacto_b200.h states the problem and the rule).  It is a local
method: from the same warm start it may stop at another local optimum than ipopt.
"""
import numpy as np
import torch

from ._lib import check, lib, ptr, stream_ptr
from .segment_tree import _dev


class TO_Casadi:
    def __init__(self, env, conf, env_TO=None, w_S=0):
        self.env = env
        self.conf = conf
        self.nx = conf.nx
        self.nu = conf.na
        self.w_S = w_S
        self.CAMS = env_TO

    def TO_System_Solve(self, *a, **k):
        raise NotImplementedError('the CasADi/ipopt solve stays on the host pool of the reference (TO.py:35-100); '
                                  'cacto_b200 provides its warm-starts (RL_AC.rollout_batch) and consumes its solutions')

    TO_Solve = TO_System_Solve

    def backward_pass_batch(self, TO_states_list, TO_controls_list, mu=1e-9):
        """TO_states_list[e]: [T_e+1, >= nx] (a trailing time column is ignored); TO_controls_list[e]: [T_e, na].
        Returns (V_x, offsets): V_x CUDA fp64 [sum(T_e+1), nx+1] over the concatenated knots (time column 0, TO.py:166)."""
        c = self.conf
        nx, na = int(c.nb_state) - 1, int(c.nb_action)
        dev = _dev()
        lens = np.array([len(s) for s in TO_states_list], dtype=np.int64)
        offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        K, E = int(offsets[-1]), len(lens)
        X = np.zeros((K, nx))
        U = np.zeros((K, na))
        for e, (s, u) in enumerate(zip(TO_states_list, TO_controls_list)):
            s = np.asarray(s, dtype=np.float64)
            u = np.asarray(u, dtype=np.float64).reshape(-1, na)
            if len(u) < len(s) - 1:
                raise ValueError('trajectory %d: %d knots need %d controls, got %d' % (e, len(s), len(s) - 1, len(u)))
            X[offsets[e]:offsets[e + 1]] = s[:, :nx]
            U[offsets[e]:offsets[e] + len(s) - 1] = u[:len(s) - 1]
        Xd, Ud = torch.as_tensor(X).to(dev), torch.as_tensor(U).to(dev)
        off_dev = torch.as_tensor(offsets).to(dev)
        return _backward_pass_packed(self.env, off_dev, E, Xd, Ud, mu), offsets

    def backward_pass(self, T, TO_states, TO_controls, mu=1e-9):
        """TO.py:119: T knots of TO_states[T, nx] and TO_controls[T-1, na] -> V_x[T, nx+1] (NumPy, like the reference)."""
        Vx, _ = self.backward_pass_batch([np.asarray(TO_states)[:T]], [np.asarray(TO_controls)[:T - 1]], mu)
        return Vx.cpu().numpy()


def _backward_pass_packed(env, off_dev, E, X, U, mu):
    """cacto_backward_pass over knots already on the device: X [K, nx], U [K, na] fp64 -> V_x [K, nx+1]."""
    K, nx = X.shape
    na = U.shape[1]
    ws = torch.empty(int(lib.cacto_backward_pass_workspace_bytes(nx, na, K)) // 8 + 1, dtype=torch.float64, device=X.device)
    Vx = torch.zeros((K, nx + 1), dtype=torch.float64, device=X.device)
    check(lib.cacto_backward_pass(env._p, ptr(off_dev), E, ptr(X), ptr(U), K, float(mu), ptr(ws), ptr(Vx), stream_ptr()), 'backward_pass')
    return Vx


class TO_DDP:
    """Batched iLQR TO solves on the GPU (kernel K7), an alternative to ``TO_Casadi.TO_Solve`` that keeps the episode on the device.

    ``solve_batch`` takes what ``RL_AC.rollout_batch`` returns and hands back what ``RL_AC.rtg_batch`` and ``buffer.add`` take."""
    RUNNING, CONVERGED, FAILED = 0, 1, 2
    N_ALPHA, HISTORY, TRAJ_DOUBLES = 8, 8, 24          # CACTO_DDP_N_ALPHA, CACTO_DDP_HISTORY, CACTO_DDP_TRAJ_DOUBLES

    def __init__(self, env, conf, check_every=4):
        self.env = env
        self.conf = conf
        self.nx, self.na, self.ns = int(conf.nb_state) - 1, int(conf.nb_action), int(conf.nb_state)
        self.check_every = int(check_every)           # iterations enqueued between two reads of the running count

    def solve_batch(self, ICS, states, controls, horizon, max_iter=100, tol=1e-8, mu_bp=1e-9):
        """ICS [E, ns]; states [T_max+1, ns, E] and controls [T_max, na, E] (fp64, the SoA layout of RL_AC.rollout_batch; CUDA
        tensors or arrays); horizon [E] (T_e = NSTEPS_SH, 0 allowed).  Trajectory e is solved over its knots 0 .. T_e from
        x_0 = ICS[e] (time column excluded).  Returns a dict:
          states, controls   solved, same layout; entries past each horizon and the time column are left as given;
          cost[E] fp64, iterations[E] int32, status[E] int32 (0 stopped at max_iter, 1 converged, 2 failed: the warm start's
                             cost is not finite or the regularisation left its range; the iterate is the best one met);
          warm_cost[E]       the warm start's cost;
          step_cost          [sum(T_e+1)] fp64 over the concatenated knots: -reward per knot, running then terminal (what
                             RL_Solve consumes as TO_step_cost);
          dVdx               [sum(T_e+1), ns] from cacto_backward_pass at the solution (mu = mu_bp);
          offsets            host int64 [E+1] of the concatenated knots;
          alpha_index[E, 8]  accepted line-search index j (alpha = 2^-j) of the first iterations, or a negative code
                             (-1 backward pass failed, -2 no step accepted, -3 converged without a step, -4 not run);
          TO_states, TO_step_cost, dVdx_list   per-episode host lists ([T_e+1, ns], [T_e+1], [T_e+1, ns]) for rtg_batch / buffer.add."""
        dev = _dev()
        nx, na, ns = self.nx, self.na, self.ns
        S_in = torch.as_tensor(states).to(dev, torch.float64)
        U_in = torch.as_tensor(controls).to(dev, torch.float64)
        T_max, E = S_in.shape[0] - 1, S_in.shape[2]
        if S_in.shape[1] != ns or U_in.shape != (T_max, na, E):
            raise ValueError('solve_batch: states [T+1, %d, E] and controls [T, %d, E] expected, got %s and %s'
                             % (ns, na, tuple(S_in.shape), tuple(U_in.shape)))
        hz = np.asarray(horizon.cpu() if isinstance(horizon, torch.Tensor) else horizon, dtype=np.int64).reshape(-1)
        if len(hz) != E or (hz < 0).any() or (hz > T_max).any():
            raise ValueError('solve_batch: horizon must hold E = %d values in [0, %d]' % (E, T_max))
        offsets = np.concatenate([[0], np.cumsum(hz + 1)]).astype(np.int64)
        K = int(offsets[-1])
        # knots of trajectory e are rows offsets[e] .. offsets[e+1]-1: a mask over (e, t) keeps that order
        mask = (torch.arange(T_max + 1, device=dev)[None, :] <= torch.as_tensor(hz, device=dev)[:, None])
        S = S_in.permute(2, 0, 1)                                            # [E, T_max+1, ns] view
        X = S[:, :, :nx].clone()
        X[:, 0] = torch.as_tensor(ICS).to(dev, torch.float64).reshape(E, ns)[:, :nx]
        X = X[mask].contiguous()
        U = torch.cat([U_in.permute(2, 0, 1), torch.zeros((E, 1, na), dtype=torch.float64, device=dev)], dim=1)[mask].contiguous()
        off_dev = torch.as_tensor(offsets).to(dev)
        ws = torch.empty(int(lib.cacto_ddp_workspace_bytes(nx, na, K, E)) // 8 + 1, dtype=torch.float64, device=dev)
        cost = torch.empty(E, dtype=torch.float64, device=dev)
        status = torch.empty(E, dtype=torch.int32, device=dev)
        iters = torch.empty(E, dtype=torch.int32, device=dev)
        p, st = self.env._p, stream_ptr()
        check(lib.cacto_ddp_init(p, ptr(off_dev), E, ptr(X), ptr(U), K, ptr(ws), ptr(cost), ptr(status), ptr(iters), st), 'ddp_init')
        warm_cost = cost.clone()
        done = 0
        while done < max_iter and E > 0:
            n = min(self.check_every, max_iter - done)
            check(lib.cacto_ddp_iterate(p, ptr(off_dev), E, ptr(X), ptr(U), K, n, float(tol), ptr(ws), ptr(cost), ptr(status), ptr(iters), st),
                  'ddp_iterate')
            done += n
            if int((status == self.RUNNING).sum()) == 0:                   # the one host read per check_every iterations
                break
        rec0 = int(lib.cacto_ddp_workspace_bytes(nx, na, K, 0)) // 8                # the per-trajectory records follow the knots
        rec = ws[rec0:rec0 + E * self.TRAJ_DOUBLES].reshape(E, self.TRAJ_DOUBLES)
        alpha_index = rec[:, 4 + self.N_ALPHA:4 + self.N_ALPHA + self.HISTORY].to(torch.int32)
        # unpack into copies of the inputs: solved knots over the warm start, the rest untouched
        S_out, U_out = S_in.clone(), U_in.clone()
        S_out.permute(2, 0, 1)[:, :, :nx][mask] = X
        last = torch.zeros(K, dtype=torch.bool, device=dev)                 # terminal knots (no control)
        last[torch.as_tensor(offsets[1:] - 1, device=dev)] = True
        U_out.permute(2, 0, 1)[mask[:, 1:]] = U[~last]                       # knot t < T_e carries a control
        S_kn = S_out.permute(2, 0, 1)[mask].contiguous()                     # [K, ns] with the time column
        w8 = torch.zeros((K, 8), dtype=torch.float64, device=dev)
        w8[:, :len(self.conf.cost_weights_running)] = torch.as_tensor(np.asarray(self.conf.cost_weights_running, dtype=np.float64), device=dev)
        w8[last, :len(self.conf.cost_weights_terminal)] = torch.as_tensor(np.asarray(self.conf.cost_weights_terminal, dtype=np.float64), device=dev)
        U_kn = torch.where(last[:, None], torch.zeros_like(U), U)
        step_cost = -self.env._reward_kernel(w8, S_kn, U_kn, False, False)[0] if K else torch.zeros(0, dtype=torch.float64, device=dev)
        dVdx = _backward_pass_packed(self.env, off_dev, E, X, U, mu_bp) if K else torch.zeros((0, ns), dtype=torch.float64, device=dev)
        S_h, c_h, v_h = S_kn.cpu().numpy(), step_cost.cpu().numpy(), dVdx.cpu().numpy()
        cut = lambda a: [a[offsets[e]:offsets[e + 1]] for e in range(E)]
        return dict(states=S_out, controls=U_out, cost=cost, warm_cost=warm_cost, iterations=iters, status=status, step_cost=step_cost,
                    dVdx=dVdx, offsets=offsets, alpha_index=alpha_index, TO_states=cut(S_h), TO_step_cost=cut(c_h), dVdx_list=cut(v_h))
