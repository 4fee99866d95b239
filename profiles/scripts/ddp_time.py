"""K7 timing: the batched iLQR TO solve (TO_DDP.solve_batch, csrc/ddp.cu) per system at the conf's EP_UPDATE trajectories and NSTEPS,
warm-started by the actor (RL_AC.rollout_batch, a freshly initialised actor, ep = 1).

Per system: ms per iteration split by kernel (torch.profiler over the first iterations of a solve),
then one full solve (max_iter = 100, tol = 1e-8) timed with CUDA events: iterations to convergence (median / max over the batch),
statuses and total ms (packing, dVdx and host lists included).  Beside it the oracle (oracle/ddp.py, NumPy on one host core): seconds
per iteration for one trajectory, and that times E as the host-side equivalent.

    python profiles/scripts/ddp_time.py [system ...]
"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from cacto_b200 import environment as genv               # noqa: E402
from cacto_b200.conf import SYSTEM_IDS, get_conf         # noqa: E402
from cacto_b200.NeuralNetwork import NN                  # noqa: E402
from cacto_b200.RL import RL_AC                          # noqa: E402
from cacto_b200.TO import TO_DDP                         # noqa: E402
from oracle import ddp as oddp                           # noqa: E402
from oracle import systems as osys                       # noqa: E402

KERNELS = ('k_ddp_knots', 'k_ddp_backward', 'k_ddp_probe', 'k_ddp_commit')


def kernel_split(ddp, ICS, states, controls, hz, n_iter=4):
    """ms per iteration per kernel over the first n_iter iterations of a solve (torch.profiler, a run of its own)."""
    ddp.solve_batch(ICS, states, controls, hz, max_iter=1)                  # warm-up
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        res = ddp.solve_batch(ICS, states, controls, hz, max_iter=n_iter)
        torch.cuda.synchronize()
    split = {k: 0.0 for k in KERNELS}
    for ev in prof.key_averages():
        for k in KERNELS:
            if k in ev.key:
                split[k] += getattr(ev, 'device_time_total', getattr(ev, 'cuda_time_total', 0.0)) / 1e3 / n_iter
    return split, int((res['status'] == ddp.RUNNING).sum())


def main(systems):
    torch.cuda.set_device(0)
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True).stdout.strip()
    print('device:', torch.cuda.get_device_name(0), '|', q, flush=True)
    for system in systems:
        conf = get_conf(system)
        env = genv.make_env(conf)
        rl = RL_AC(env, NN(env, conf, 1e-2, seed=0), conf, 0)
        rl.setup_model()
        E, T = int(conf.EP_UPDATE), int(conf.NSTEPS)
        rng = np.random.default_rng(0)
        ICS = rng.uniform(np.asarray(conf.x_init_min, float), np.asarray(conf.x_init_max, float), (E, conf.nb_state))
        ICS[:, -1] = 0.0                                                    # full horizon: NSTEPS_SH = NSTEPS
        out = rl.rollout_batch(ICS, 1)
        hz = out['horizon'].cpu().numpy()
        ddp = TO_DDP(env, conf)
        split, running = kernel_split(ddp, ICS, out['states'], out['controls'], hz)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        res = ddp.solve_batch(ICS, out['states'], out['controls'], hz, max_iter=100, tol=1e-8)
        e1.record()
        torch.cuda.synchronize()
        total = e0.elapsed_time(e1)
        iters = res['iterations'].cpu().numpy()
        status = res['status'].cpu().numpy()
        gain = 1 - res['cost'].cpu().numpy() / res['warm_cost'].cpu().numpy()
        # the oracle, one trajectory, one iteration
        oenv = osys.make_env(conf)
        U0 = out['controls'][:, :, 0].cpu().numpy()
        t0 = time.perf_counter()
        o = oddp.solve(oenv, ICS[0, :-1], U0, max_iter=1, tol=0.0)
        t_or = (time.perf_counter() - t0) / max(1, o['iterations'])
        per_it = sum(split.values())
        print('%-17s E=%d T=%d  per iteration (first 4; %d still running after them): %.3f ms = %s' % (
            system, E, T, running, per_it, ' + '.join('%s %.3f' % (k[6:], v) for k, v in split.items())), flush=True)
        print('%-17s solve: %.1f ms total, iterations median %d max %d, status converged %d / failed %d / max_iter %d, '
              'median cost reduction %.1f %%' % (system, total, int(np.median(iters)), int(iters.max()), (status == 1).sum(),
                                                  (status == 2).sum(), (status == 0).sum(), 100 * np.median(gain)), flush=True)
        print('%-17s oracle (NumPy, 1 host core): %.2f s per iteration per trajectory -> %.0f s per iteration for E=%d' % (
            system, t_or, t_or * E, E), flush=True)


if __name__ == '__main__':
    main(sys.argv[1:] or SYSTEM_IDS)
