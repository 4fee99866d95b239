"""Width-generic actor kernels (csrc/actor_width.cu) against the fused 256-wide engines, on one GPU in one process.

  rollouts: manipulator, 131 072 rollouts x 100 steps (BASELINE config 3), L2 overwritten before every timed pass; the width-generic
            kernel at widths 64 / 128 / 256 / 512, alternating with the fused 'fma' and 'tc' engines at 256.  Env-steps/s and the
            actor's share of the FP32 FMA peak measured in the same run (cacto_peak_fma_fp32).
  updates:  one RL_AC update replayed as a CUDA graph (UpdateGraph) and as the pipelined graph (PipelinedUpdateGraph, where it
            applies), manipulator, B = 64 and 4096, the same widths; at 256 the fused path.

usage: python profiles/scripts/actor_width_time.py [out.json]
"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from cacto_b200 import environment as genv                      # noqa: E402
from cacto_b200._lib import check, lib, ptr, stream_ptr          # noqa: E402
from cacto_b200.conf import get_conf                             # noqa: E402
from cacto_b200.ops import ops                                   # noqa: E402
from cacto_b200.NeuralNetwork import NN                          # noqa: E402
from cacto_b200.RL import RL_AC                                  # noqa: E402

WIDTHS = (64, 128, 256, 512)


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def fma_peak():
    out = torch.zeros(1, device='cuda')
    blocks, iters = 148 * 16, 20000
    check(lib.cacto_peak_fma_fp32(ptr(out), iters, blocks, stream_ptr()), 'peak')
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(lib.cacto_peak_fma_fp32(ptr(out), iters, blocks, stream_ptr()), 'peak')
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) * 1e-3)
    return blocks * 256 * iters * 16 * 2 / best


def build(widths, **over):
    conf = get_conf('manipulator', NH1=widths[0], NH2=widths[1], **over)
    env = genv.make_env(conf)
    nn = NN(env, conf, 1e-2, seed=0)
    rl = RL_AC(env, nn, conf, 0)
    rl.setup_model()
    return conf, nn, rl


def rollouts(peak):
    B, T = 131072, 100
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    cases = [('width', w) for w in WIDTHS] + [('fma', 256), ('tc', 256)]
    runs = {}
    for eng, w in cases:
        conf, nn, rl = build((w, w), NSTEPS=T)
        rng = np.random.default_rng(0)
        x = rng.uniform(np.asarray(conf.x_init_min, float), np.asarray(conf.x_init_max, float), (B, conf.nb_state))
        x[:, -1] = 0.0
        ics = torch.as_tensor(x, device='cuda')
        hz = torch.full((B,), T, dtype=torch.int32, device='cuda')
        st = torch.empty((T + 1) * conf.nb_state * B, dtype=torch.float64, device='cuda').view(T + 1, conf.nb_state, B)
        ct = torch.empty(T * conf.nb_action * B, dtype=torch.float64, device='cuda').view(T, conf.nb_action, B)
        fl = torch.empty(B, dtype=torch.int32, device='cuda')
        runs[(eng, w)] = (rl, conf, ics, hz, st, ct, fl)
    times = {k: [] for k in runs}
    for rep in range(6):                                          # alternate the engines; the first pass of each warms up
        for k, (rl, conf, ics, hz, st, ct, fl) in runs.items():
            flush.fill_(rep & 0xff)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            if k[0] == 'width':                                   # the op directly: a 256-wide actor would take the fused engines
                ops.rollout_width(rl.env._pt, rl.actor_model.params, k[1], k[1], ics, hz, T, st, ct, fl, None)
            else:
                rl._launch_rollout(1, ics, hz, T, st, ct, fl, None, B, engine=k[0])
            e1.record()
            torch.cuda.synchronize()
            assert bool(fl.all()), k
            if rep:
                times[k].append(e0.elapsed_time(e1) * 1e-3)
    out = []
    for (eng, w), ts in times.items():
        conf = runs[(eng, w)][1]
        t = float(np.median(ts))
        flops = 2.0 * (conf.nb_state * w + w * w + w * conf.nb_action) * B * T
        out.append(dict(engine=eng if eng != 'width' else 'width-generic', width=w, ms=t * 1e3, ms_min=min(ts) * 1e3, ms_max=max(ts) * 1e3,
                        env_steps_per_s=B * T / t, actor_fma_share_of_peak=flops / t / peak))
        print('rollout %-13s %3d: %8.2f ms (min %.2f max %.2f)  %.3g env-steps/s  actor %.1f %% of FP32 FMA peak' %
              (out[-1]['engine'], w, t * 1e3, min(ts) * 1e3, max(ts) * 1e3, B * T / t, 100 * flops / t / peak), flush=True)
    return out


def updates():
    out = []
    for B in (64, 4096):
        for w in WIDTHS:
            conf, nn, rl = build((w, w), BATCH_SIZE=B)
            rng = np.random.default_rng(1)
            ns = conf.nb_state
            lo, hi = np.asarray(conf.x_init_min, float), np.asarray(conf.x_init_max, float)
            data = dict(state=rng.uniform(lo, hi, (B, ns)), state_next=rng.uniform(lo, hi, (B, ns)), partial_rtg=rng.uniform(-5, 0, (B, 1)),
                        dVdx=rng.normal(size=(B, ns)), done=(rng.uniform(size=(B, 1)) < 0.5) * 1.0, term=(rng.uniform(size=(B, 1)) < 0.2) * 1.0,
                        weights=rng.uniform(0.2, 1.5, (B, 1)))
            row = dict(B=B, width=w, actor=rl.actor_model.kind)
            makers = [('graph', rl.make_update_graph)]
            if not nn._use_tc(B):
                makers.append(('pipelined', rl.make_pipelined_update_graph))
            for name, mk in makers:
                g = mk(B)
                for k, v in data.items():
                    g.io[k].copy_(torch.as_tensor(v).reshape(g.io[k].shape))
                for _ in range(20):
                    g.replay()
                torch.cuda.synchronize()
                best = 1e9
                for _ in range(5):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(100):
                        g.replay()
                    e1.record()
                    torch.cuda.synchronize()
                    best = min(best, e0.elapsed_time(e1) * 1e3 / 100)
                if hasattr(g, 'flush'):
                    g.flush()
                row[name + '_us'] = best
            out.append(row)
            print('update B=%5d width %3d (%s): %s' % (B, w, row['actor'], ', '.join('%s %.1f us' % (k[:-3], v) for k, v in row.items() if k.endswith('_us'))),
                  flush=True)
    return out


def main():
    info = gpu_info()
    print('GPU:', info, flush=True)
    peak = fma_peak()
    print('FP32 FMA peak (in-run): %.1f TFLOP/s' % (peak / 1e12), flush=True)
    res = dict(gpu=info, fma_peak_flops=peak, rollouts=rollouts(peak), updates=updates())
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
        with open(sys.argv[1], 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
