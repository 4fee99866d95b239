"""Child process of tests/test_gpu_deterministic.py::test_simulated_ranks_are_bit_identical: two simulated peer-memory ranks on one
GPU (as tests/peer_sim_check.py) with NN(..., deterministic=True), the static launch sequence of the update graph, run twice from
the same seed.  The replicas must be bit-identical within a run and the runs bit-identical to each other.  Prints 'peer-sim-det ok'."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from test_gpu_peer_reduce import IO_KEYS, SimDist, batch, flat


def make_rl(system, dist, region):
    from cacto_b200 import environment as genv
    from cacto_b200.NeuralNetwork import NN
    from cacto_b200.RL import RL_AC
    from cacto_b200.conf import get_conf
    conf = get_conf(system)
    env = genv.make_env(conf)
    rl = RL_AC(env, NN(env, conf, 1e-2, seed=0, deterministic=True), conf, 0, dist=dist, peer_region=region, peer_max_ctas=16)
    rl.setup_model()
    return conf, rl


def run(system='manipulator', world=2, Bl=16):
    from cacto_b200.parallel import PeerReduce, PeerRegion
    conf, probe = make_rl(system, None, None)
    # one update on the same batch size first: it loads the deterministic kernels, so that no lazy module load (which may wait for
    # the device) happens while a rank's peer kernel waits for the other rank's launches
    probe.update(*[batch(conf, Bl, 0)[k] for k in IO_KEYS], fuse_target=True)
    torch.cuda.synchronize()
    regions = PeerRegion.local_group(PeerReduce.region_bytes(probe.critic_model.n, probe.actor_model.n), world)
    ranks = [make_rl(system, SimDist(r, world), regions[r])[1] for r in range(world)]
    assert all(rl._peer is not None for rl in ranks)
    streams = [torch.cuda.Stream() for _ in range(world)]
    ios = []
    for r in range(world):
        with torch.cuda.stream(streams[r]):
            io = batch(conf, Bl, 0)
            io.update(rtg=torch.zeros((Bl, 1), device='cuda'), V=torch.zeros((Bl, 1), device='cuda'), V_target=torch.zeros((Bl, 1), device='cuda'))
            ios.append(io)
            for o, n in ((ranks[r].critic_optimizer, ranks[r].critic_model), (ranks[r].actor_optimizer, ranks[r].actor_model)):
                o.moments(n)
                o._device_state(n.params.device)
            ranks[r].NN._det_partials(ranks[r].NN.DET_CRITIC, Bl)      # the partials workspaces, allocated on the rank's stream
            ranks[r].NN._det_partials(ranks[r].NN.DET_ACTOR, Bl)
            scratch = [torch.empty((Bl, 1), device='cuda') for _ in range(8)] + [torch.empty((Bl, conf.nb_state), device='cuda') for _ in range(8)]
            del scratch
    torch.cuda.synchronize()
    for it in range(3):
        g = batch(conf, Bl * world, 10 + it)
        for r in range(world):
            for k in IO_KEYS:
                ios[r][k].copy_(g[k][r * Bl:(r + 1) * Bl])
        torch.cuda.synchronize()
        for r, rl in enumerate(ranks):
            with torch.cuda.stream(streams[r]):
                rl._update_static(ios[r])
        torch.cuda.synchronize()
    out = [flat(rl) for rl in ranks]
    for rg in regions:
        rg.close()
    return out


if __name__ == '__main__':
    a, b = run(), run()
    assert torch.equal(a[0], a[1]) and torch.equal(b[0], b[1]), 'replicas must stay bit-identical'
    assert torch.equal(a[0], b[0]), 'two runs of the same seeded update differ'
    print('peer-sim-det ok', flush=True)
