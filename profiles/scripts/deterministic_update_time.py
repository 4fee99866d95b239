"""Device time per update, NN(deterministic=True) against the default path, as a replayed CUDA graph (UpdateGraph) and, where it
applies, pipelined (PipelinedUpdateGraph).  Both paths pick the same engine: the fused FMA kernels below B = 2400 (NN.TC_MIN_BATCH),
the tcgen05 kernels from there, where the pipelined graph does not apply.  Run from the repository root on a GPU."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

import subprocess

import torch

from cacto_b200 import environment as genv
from cacto_b200.NeuralNetwork import NN
from cacto_b200.RL import RL_AC
from cacto_b200.conf import get_conf
from cacto_b200.replay_buffer import ReplayBuffer
from test_gpu_update_graph import fill


def build(system, B, deterministic):
    conf = get_conf(system, BATCH_SIZE=B)
    env = genv.make_env(conf)
    rl = RL_AC(env, NN(env, conf, 1e-2, seed=0, deterministic=deterministic), conf, 0)
    rl.setup_model()
    return conf, rl


def dev_time(g, n):
    for _ in range(10):
        g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n * 1e3


def main():
    if not torch.cuda.is_available():
        raise SystemExit('needs a GPU')
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True).stdout.strip()
    print('GPU:', q, flush=True)
    for system, B in (('manipulator', 64), ('ur5', 64), ('manipulator', 4096), ('manipulator', 16384)):
        n = 400 if B <= 128 else 60
        row = {}
        for det in (False, True):
            conf, rl = build(system, B, det)
            buf = ReplayBuffer(conf)
            fill(buf, conf, 60000)
            g = rl.make_update_graph(B)
            buf.sample(out=g.io)
            row[('graph', det)] = dev_time(g, n)
            if not rl.NN._use_tc(B):
                p = rl.make_pipelined_update_graph(B)
                buf.sample(out=p.ios[0])
                buf.sample(out=p.ios[1])
                row[('pipelined', det)] = dev_time(p, n)
                p.flush()
            del g, rl, buf
            torch.cuda.synchronize()
        fmt = lambda k: f"{row[k]:.1f}" if k in row else '-'
        print(f"{system} B={B}: graph {fmt(('graph', False))} us default, {fmt(('graph', True))} us deterministic; "
              f"pipelined {fmt(('pipelined', False))} us default, {fmt(('pipelined', True))} us deterministic", flush=True)


if __name__ == '__main__':
    main()
