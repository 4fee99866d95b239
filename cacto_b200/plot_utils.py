"""plot_utils.py of the reference, the part that is on the hot path: ``PLOT.rollout`` (plot_utils.py:245-279) -- the second caller of
the fused actor + dynamics rollout (SURVEY.md 8f4): evaluation rollouts of an actor from conf.init_states_sim with the running
reward of every step.  All rollouts run in ONE launch of the rollout kernel (torch.ops.cacto.rollout with its reward output) and
one batched forward-kinematics launch; the matplotlib figures of the reference are out of scope (SURVEY.md section 2, row 13):
``plot_policy_eval`` only keeps the data the reference would draw."""
import numpy as np
import torch

from .environment import _as_cuda, _device
from .ops import ops


class PLOT:
    """plot_utils.py:9-45: PLOT(N_try, env, NN, conf)."""

    def __init__(self, N_try, env, NN, conf):
        self.env = env
        self.NN = NN
        self.conf = conf
        self.N_try = N_try
        self.p_ee_all_sim = None           # what plot_policy_eval received last

    def rollout(self, update_step_cntr, actor_model, init_states_sim, diff_loc=0):
        """plot_utils.py:245-279.  For every initial state: NSTEPS steps of ``u = actor(x)``, ``x', r = env.step(w_running, x, u)``
        (no early stop, no NaN check -- as the reference); the EE path with its z column replaced by the third state component from
        the second knot on (:266, quirk kept); returns {(x0, y0): episodic reward}, the sum of the NSTEPS running rewards."""
        c = self.conf
        dev = _device()
        ics = _as_cuda(np.asarray(init_states_sim, dtype=np.float64), torch.float64).reshape(-1, c.nb_state)
        B, T, ns, na = ics.shape[0], int(c.NSTEPS), int(c.nb_state), int(c.nb_action)
        hz = torch.full((B,), T, dtype=torch.int32, device=dev)
        states = torch.empty((T + 1, ns, B), dtype=torch.float64, device=dev)
        controls = torch.empty((T, na, B), dtype=torch.float64, device=dev)
        flags = torch.empty(B, dtype=torch.int32, device=dev)
        rewards = torch.empty((T + 1, B), dtype=torch.float64, device=dev)
        # the fp32 CUDA-core engines: a handful of rollouts, no fp16 range limit
        if actor_model.kind == 'actor_width':
            ops.rollout_width(self.env._pt, actor_model.params, actor_model.dims[1], actor_model.dims[2], ics, hz, T, states, controls, flags, rewards)
        else:
            ops.rollout(self.env._pt, actor_model.params, 1, ics, hz, T, states, controls, flags, rewards)
        per_rollout = states.permute(2, 0, 1).contiguous()                       # [B, T+1, ns]
        p_ee = torch.empty((B * (T + 1), 3), dtype=torch.float64, device=dev)
        ops.ee_position(self.env._pt, 0, per_rollout.reshape(-1, ns), p_ee)
        p_ee = p_ee.reshape(B, T + 1, 3)
        p_ee[:, 1:, 2] = per_rollout[:, 1:, 2]                                   # plot_utils.py:266
        p_ee_h, rew_h = p_ee.cpu().numpy(), rewards[:T].cpu().numpy()
        self.rollout_states = per_rollout.cpu().numpy()
        self.rollout_controls = controls.permute(2, 0, 1).cpu().numpy()
        init = np.asarray(init_states_sim, dtype=np.float64).reshape(-1, ns)
        returns, p_ee_all_sim = {}, []
        for k in range(B):
            ep_reward = 0
            for i in range(T):                                                   # the reference's summation order
                ep_reward += rew_h[i, k]
            if k == 0:
                print("N try = {}: Simulation Return @ N updates = {} ==> {}".format(self.N_try, update_step_cntr, ep_reward))
            p_ee_all_sim.append(p_ee_h[k])
            returns[init[k][0], init[k][1]] = ep_reward
        self.plot_policy_eval(p_ee_all_sim, update_step_cntr, diff_loc=diff_loc)
        return returns

    def plot_policy_eval(self, p_list, n_updates, diff_loc=0, PRETRAIN=0):
        """plot_utils.py:186-243 draws the EE paths; here the data is kept (figures are out of scope)."""
        self.p_ee_all_sim = p_list
