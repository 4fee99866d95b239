"""Host-side mirror of the reference's ``RL.py`` (class ``RL_AC``) on the CUDA hot path.

  setup_model        RL.py:61-99    networks + Adam (+ PiecewiseConstantDecay when conf.LR_SCHEDULE)
  update             RL.py:101-111  critic gradient -> Adam, then actor gradient (with the UPDATED critic) -> Adam
  update_target      RL.py:113-118  Polyak averaging
  learn_and_update   RL.py:120-143  sample -> update -> priorities -> target
  RL_Solve           RL.py:145-189  n-step reward-to-go of one TO trajectory (kernel K5)
  create_TO_init     RL.py:197-233  policy rollout warm-start of one initial condition (kernel K1)
plus the batched entry points the reference lacks and the metric needs:
  rollout_batch(ICS[B, ns], ep)     all warm-starts of an episode batch in one launch
  rtg_batch(...)                    all reward-to-go windows of an episode batch in one launch
Data parallelism (``dist`` = an initialised torch.distributed group): each rank passes its shard of the
minibatch, gradients are summed with one NCCL all-reduce per network before the Adam step
(critic and actor steps are sequentially dependent, RL.py:104-109).
"""
import numpy as np
import torch

from ._lib import check, lib, ptr, stream_ptr
from .environment import _as_cuda, _device
from .ops import ops
from .optim import Adam, PiecewiseConstantDecay
from .parallel import PeerReduce, PeerRegion, PeerUnavailable, allreduce_sum
from .rtg import rtg_batch as _rtg_batch

TC16_MAX_NS = 8          # inputs the fp16 rollout kernel holds: T16_MAX_NS = 8 in csrc/rollout_tc16.cu


class CompactRollouts:
    """The reference-shaped view of a ``rollout_to_host(..., compact=True)`` batch: ``states(b)`` -> [T_b+1, ns] float64 with the
    time column rebuilt by repeated addition (bit-identical to what the kernel integrates), ``controls(b)`` -> [T_b, na] float64."""

    def __init__(self, conf, ics_host, states_host, controls_host, horizon):
        self.dt = float(conf.dt)
        self.t0 = np.asarray(ics_host)[:, -1].astype(np.float64)
        self.states_host, self.controls_host, self.horizon = states_host.numpy(), controls_host.numpy(), np.asarray(horizon)

    def states(self, b):
        T = int(self.horizon[b])
        out = np.empty((T + 1, self.states_host.shape[1] + 1))
        out[:, :-1] = self.states_host[:T + 1, :, b]
        t = np.full(T + 1, self.dt)
        t[0] = self.t0[b]
        out[:, -1] = np.add.accumulate(t)                        # t_{k+1} = t_k + dt, sequentially, as the kernel does
        return out

    def controls(self, b):
        return self.controls_host[:int(self.horizon[b]), :, b].astype(np.float64)


class RL_AC:
    def __init__(self, env, NN, conf, N_try, dist=None, reduce='peer', peer_region=None, peer_max_ctas=0):
        """``dist``: the initialised ``torch.distributed`` module (or an object with its get_rank / get_world_size / broadcast
        surface) for the data-parallel update over the GPUs of one box; ``reduce``: 'peer' sums the gradient blocks over NVLink
        peer memory inside the Adam kernel (parallel.PeerReduce), 'nccl' launches one all-reduce per network before it;
        ``peer_region``: a ready ``PeerRegion`` (tests simulate several ranks on one GPU with ``PeerRegion.local_group``)."""
        self.env = env
        self.NN = NN
        self.conf = conf
        self.N_try = N_try
        self.dist = dist
        if reduce not in ('peer', 'nccl'):
            raise ValueError('unknown gradient reduction %r' % (reduce,))
        self.reduce = reduce
        self._peer_region, self._peer_max_ctas = peer_region, peer_max_ctas
        self._peer = None

        self.actor_model = None
        self.critic_model = None
        self.target_critic = None
        self.actor_optimizer = None
        self.critic_optimizer = None

        self.init_rand_state = None
        self.NSTEPS_SH = 0
        self.control_arr = None
        self.state_arr = None
        self.ee_pos_arr = None
        self.exp_counter = np.zeros(conf.REPLAY_SIZE)

    # ------------------------------------------------------------------------------ models
    def setup_model(self, recover_training=None):
        """RL.py:61-99."""
        c = self.conf
        self.actor_model = self.NN.create_actor()
        if c.critic_type == 'sine':
            self.critic_model = self.NN.create_critic_sine()
            self.target_critic = self.NN.create_critic_sine()
        elif c.critic_type == 'elu':
            self.critic_model, self.target_critic = self.NN.create_critic_elu(), self.NN.create_critic_elu()
        elif c.critic_type == 'sine-elu':
            self.critic_model, self.target_critic = self.NN.create_critic_sine_elu(), self.NN.create_critic_sine_elu()
        else:
            self.critic_model, self.target_critic = self.NN.create_critic_relu(), self.NN.create_critic_relu()

        if c.LR_SCHEDULE:
            self.CRITIC_LR_SCHEDULE = PiecewiseConstantDecay(c.boundaries_schedule_LR_C, c.values_schedule_LR_C)
            self.ACTOR_LR_SCHEDULE = PiecewiseConstantDecay(c.boundaries_schedule_LR_A, c.values_schedule_LR_A)
            self.critic_optimizer = Adam(self.CRITIC_LR_SCHEDULE)
            self.actor_optimizer = Adam(self.ACTOR_LR_SCHEDULE)
        else:
            self.critic_optimizer = Adam(c.CRITIC_LEARNING_RATE)
            self.actor_optimizer = Adam(c.ACTOR_LEARNING_RATE)

        if recover_training is not None:
            path, n_try, step = str(recover_training[0]), recover_training[1], recover_training[2]
            # the reference's archive layout (RL.py:95-97): <path>/N_try_<n>/<net>_<step>.h5; Network.load_weights falls back to
            # the .npz of the same stem when no .h5 is there
            self.actor_model.load_weights("{}/N_try_{}/actor_{}.h5".format(path, n_try, step))
            self.critic_model.load_weights("{}/N_try_{}/critic_{}.h5".format(path, n_try, step))
            self.target_critic.load_weights("{}/N_try_{}/target_critic_{}.h5".format(path, n_try, step))
        else:
            self.target_critic.set_weights(self.critic_model.get_weights())
        if self.dist is not None:                       # identical replicas: broadcast rank 0's initial weights
            for net in (self.actor_model, self.critic_model, self.target_critic):
                self.dist.broadcast(net.params, src=0)
                net.refresh_transposed()
            if self.reduce == 'peer' and self.dist.get_world_size() > 1 and self.actor_model.params.is_cuda:
                region = self._peer_region
                if region is None:
                    try:
                        region = PeerRegion.exchange(PeerReduce.region_bytes(self.critic_model.n, self.actor_model.n), self.dist)
                    except PeerUnavailable as e:         # unanimous across ranks: every rank takes the NCCL all-reduce instead
                        import warnings
                        warnings.warn('peer-memory gradient exchange unavailable (%s): using NCCL all-reduce' % e)
                if region is not None:
                    self._peer = PeerReduce(region, self.critic_model, self.actor_model, max_ctas=self._peer_max_ctas)

    # ------------------------------------------------------------------------------ update
    def _reduce_and_step(self, opt, net, other, target=None, tau=0.0, prepared=False):
        """Sum the per-rank gradient blocks (each rank used 1/global_batch) and apply the Adam step: one kernel over NVLink
        peer memory, or an NCCL all-reduce followed by the single-GPU kernel."""
        if self._peer is not None:
            opt.step(net, target=target, tau=tau, prepared=prepared, peer=self._peer.table(net), zero_other=other.grad)
        else:
            allreduce_sum(net.grad, self.dist)
            opt.step(net, target=target, tau=tau, prepared=prepared)

    def peer_barrier(self):
        """Host-level rendezvous of the data-parallel ranks before a run of peer-memory updates.  k_adam_peer spins on the
        arrival flags of its peers and traps after 20 s; in the CACTO loop the ranks reach the update phase after host-side TO
        solves whose duration differs per rank by far more than that, so the skew is absorbed HERE (an NCCL barrier blocks the
        host, not a kernel): afterwards all ranks launch their updates in lock-step.  No-op without the peer exchange."""
        barrier = getattr(self.dist, 'barrier', None)    # ranks simulated inside one process (tests) have nothing to wait for
        if self._peer is not None and barrier is not None:
            torch.cuda.current_stream().synchronize()
            barrier()

    def update(self, state_batch, state_next_rollout_batch, partial_reward_to_go_batch, dVdx_batch, d_batch, term_batch, weights_batch,
               batch_size=None, fuse_target=False, synced=False):
        """RL.py:101-111.  ``fuse_target`` additionally performs update_target inside the critic's Adam launch
        (used by learn_and_update; the target is only read again at the next critic gradient, so the result is
        identical to calling update_target afterwards).  ``synced``: the caller has already called ``peer_barrier`` for this
        run of updates (learn_and_update does, once per call)."""
        if not synced:
            self.peer_barrier()
        world = self.dist.get_world_size() if self.dist is not None else 1
        gb = state_batch.shape[0] * world
        # the learning-rate schedules / step counters of both Adam steps in one launch (every launch on this path is ~3 us)
        type(self.critic_optimizer).prepare_pair(self.critic_optimizer, self.actor_optimizer, self.critic_model.params.device)
        critic_grad, reward_to_go_batch, critic_value, target_critic_value = self.NN.compute_critic_grad(
            self.critic_model, self.target_critic, state_batch, state_next_rollout_batch, partial_reward_to_go_batch, dVdx_batch, d_batch,
            weights_batch, global_batch=gb)
        if world > 1:
            fused = fuse_target and not self.conf.MC
            self._reduce_and_step(self.critic_optimizer, self.critic_model, self.actor_model, self.target_critic if fused else None,
                                  self.conf.UPDATE_RATE if fused else 0.0, prepared=True)
        elif fuse_target and not self.conf.MC:
            self.critic_optimizer.step(self.critic_model, target=self.target_critic, tau=self.conf.UPDATE_RATE, prepared=True)
        else:
            self.critic_optimizer.apply_gradients(zip(critic_grad, self.critic_model.trainable_variables), prepared=True)

        actor_grad = self.NN.compute_actor_grad(self.actor_model, self.critic_model, state_batch, term_batch, batch_size, global_batch=gb)
        if world > 1:
            self._reduce_and_step(self.actor_optimizer, self.actor_model, self.critic_model, prepared=True)
        else:
            self.actor_optimizer.apply_gradients(zip(actor_grad, self.actor_model.trainable_variables), prepared=True)
        return reward_to_go_batch, critic_value, target_critic_value

    # ------------------------------------------------------------------------------ CUDA-graph update
    def _update_static(self, io):
        """The launches of one update + target update on pre-allocated tensors (no allocation, no host scalars):
        what ``make_update_graph`` captures.  Gradient accumulators are left zeroed by the Adam kernel."""
        c, nn = self.conf, self.NN
        world = self.dist.get_world_size() if self.dist is not None else 1
        B = io['state'].shape[0]
        inv_B = 1.0 / float(B * world)
        cm, tc, am = self.critic_model, self.target_critic, self.actor_model
        type(self.critic_optimizer).prepare_pair(self.critic_optimizer, self.actor_optimizer, cm.params.device, zero=nn.last_critic_loss)
        nn.launch_critic_grad(cm, tc, io['state'], io['state_next'], io['partial_rtg'], io['dVdx'], io['done'], io['weights'], inv_B,
                              io['rtg'], io['V'], io['V_target'], B)
        if c.MC:
            self._reduce_and_step(self.critic_optimizer, cm, am, prepared=True)
        else:
            self._reduce_and_step(self.critic_optimizer, cm, am, target=tc, tau=c.UPDATE_RATE, prepared=True)
        nn.launch_actor_grad(am, cm, io['state'], io['term'], inv_B, None, B)
        self._reduce_and_step(self.actor_optimizer, am, cm, prepared=True)

    def _critic_step_static(self, io, schedule=True):
        """Critic half of ``_update_static`` (schedule, gradient, Adam + Polyak) on the tensors of ``io``."""
        c, nn = self.conf, self.NN
        B = io['state'].shape[0]
        cm, tc, am = self.critic_model, self.target_critic, self.actor_model
        if schedule:
            self.critic_optimizer.prepare(cm.params.device, zero=nn.last_critic_loss)
        nn.launch_critic_grad(cm, tc, io['state'], io['state_next'], io['partial_rtg'], io['dVdx'], io['done'], io['weights'], 1.0 / float(B),
                              io['rtg'], io['V'], io['V_target'], B)
        if c.MC:
            self._reduce_and_step(self.critic_optimizer, cm, am, prepared=True)
        else:
            self._reduce_and_step(self.critic_optimizer, cm, am, target=tc, tau=c.UPDATE_RATE, prepared=True)

    def _actor_step_static(self, io, schedule=True):
        """Actor half of ``_update_static`` (schedule, gradient through the -- already updated -- critic, Adam)."""
        B = io['state'].shape[0]
        am, cm = self.actor_model, self.critic_model
        if schedule:
            self.actor_optimizer.prepare(am.params.device)
        self.NN.launch_actor_grad(am, cm, io['state'], io['term'], 1.0 / float(B), None, B)
        self._reduce_and_step(self.actor_optimizer, am, cm, prepared=True)

    def make_pipelined_update_graph(self, batch_size=None):
        """``PipelinedUpdateGraph``: consecutive updates overlapped on one GPU (critic step of batch i beside the actor step of batch
        i - 1; same results as the sequential order).  Single-GPU, fused 'sine' engine only."""
        return PipelinedUpdateGraph(self, int(batch_size or self.conf.BATCH_SIZE))

    def make_update_graph(self, batch_size=None):
        """Capture update + update_target for a fixed batch size into a CUDA graph.  Returns an ``UpdateGraph`` whose
        ``io`` tensors (state, state_next, partial_rtg, dVdx, done, term, weights -> rtg, V, V_target) are filled by
        ``buffer.sample(out=graph.io)`` and whose ``replay()`` performs one update; training state is untouched by the capture."""
        return UpdateGraph(self, int(batch_size or self.conf.BATCH_SIZE))

    def update_target(self, target_weights, weights):
        """RL.py:113-118: a <- b * tau + a * (1 - tau)."""
        tau = float(self.conf.UPDATE_RATE)
        for a, b in zip(target_weights, weights):
            a.copy_(b * tau + a * (1 - tau))

    def learn_and_update(self, update_step_counter, buffer, ep):
        """RL.py:120-143."""
        self.peer_barrier()                             # data-parallel ranks arrive here with minutes of skew (host TO solves)
        graph = getattr(self, 'update_graph', None)
        world = self.dist.get_world_size() if self.dist is not None else 1
        # the update as a replayed CUDA graph (built once per batch size): at the conf batches it is launch-latency bound.  With the
        # NCCL all-reduce fallback (no peer memory) the update stays eager: a collective inside a capture ties the graph to the communicator
        # On one GPU with the fused 'sine' engine consecutive updates are software-pipelined (PipelinedUpdateGraph: same weights,
        # 1.6 x the updates/s at the conf batches); the outstanding actor step is flushed before a checkpoint and on return.
        def make():
            B = int(self.conf.BATCH_SIZE)
            if self.use_pipelined_updates and world == 1 and self.critic_model.kind == 'critic_sine' and not self.NN._use_tc(B):
                return self.make_pipelined_update_graph(B)
            return self.make_update_graph(B)
        if graph is None and self.use_update_graph and (world == 1 or self._peer is not None):
            graph = self.update_graph = make()
        if graph is not None and graph.B != int(self.conf.BATCH_SIZE):
            graph = self.update_graph = make()
        flush = getattr(graph, 'flush', None)
        loops = int(self.conf.UPDATE_LOOPS[ep])
        # uniform buffer: the index draws of the loop in a few np.random calls and copies (same stream, ReplayBuffer.index_stream)
        rows = buffer.index_stream(loops) if graph is not None and hasattr(buffer, 'index_stream') else iter(lambda: None, 0)
        for k in range(loops):
            if graph is not None:                       # captured update: the sampled rows land in the graph's input tensors
                batch_idxes = buffer.sample(next(rows), out=graph.io)[7]
                reward_to_go_batch, critic_value, target_critic_value = graph.replay()
            else:
                state_batch, partial_reward_to_go_batch, state_next_rollout_batch, dVdx_batch, d_batch, term_batch, weights_batch, batch_idxes = buffer.sample()
                reward_to_go_batch, critic_value, target_critic_value = self.update(
                    state_batch, state_next_rollout_batch, partial_reward_to_go_batch, dVdx_batch, d_batch, term_batch, weights_batch,
                    fuse_target=True, synced=True)
            if self.conf.prioritized_replay_alpha != 0:
                buffer.update_priorities(batch_idxes, reward_to_go_batch, critic_value, target_critic_value)
            update_step_counter += 1
            if update_step_counter % self.conf.save_interval == 0:
                if flush is not None:
                    flush()
                self.RL_save_weights(update_step_counter)
        if flush is not None:
            flush()
        return update_step_counter

    def RL_save_weights(self, update_step_counter='final'):
        """RL.py:191-195: <NNs_path>/N_try_<n>/{actor,critic,target_critic}_<step>.h5 (Keras save_weights files)."""
        import os
        d = self.conf.NNs_path + "/N_try_{}".format(self.N_try)
        os.makedirs(d, exist_ok=True)
        self.actor_model.save_weights(d + "/actor_{}.h5".format(update_step_counter))
        self.critic_model.save_weights(d + "/critic_{}.h5".format(update_step_counter))
        self.target_critic.save_weights(d + "/target_critic_{}.h5".format(update_step_counter))

    # ------------------------------------------------------------------------------ reward-to-go
    def rtg_batch(self, TO_states_list, TO_step_cost_list, lengths=None):
        return _rtg_batch(self.conf, TO_states_list, TO_step_cost_list, lengths)

    def RL_Solve(self, TO_controls, TO_states, TO_step_cost):
        """RL.py:145-189: returns the reference's 9-tuple (NumPy).  env_RL = 0 (every conf) takes states and rewards from the
        TO solution (:168); env_RL = 1 re-simulates the TO controls through Env.step from the stored initial state (:159-166)."""
        self.control_arr = TO_controls
        if self.conf.env_RL:
            T = self.NSTEPS_SH
            rwrd_arr = np.empty(T + 1)
            for k in range(T):
                self.state_arr[k + 1, :], rwrd_arr[k] = self.env.step(self.conf.cost_weights_running, self.state_arr[k, :], self.control_arr[k, :])
                self.ee_pos_arr[k + 1, :] = self.env.get_end_effector_position(self.state_arr[k + 1, :])
            rwrd_arr[-1] = self.env.reward(self.conf.cost_weights_terminal, self.state_arr[-1, :])
            TO_states, TO_step_cost = self.state_arr, -rwrd_arr
        out = _rtg_batch(self.conf, [TO_states], [TO_step_cost])
        self.state_arr = np.asarray(TO_states)
        rwrd_arr = -np.asarray(TO_step_cost, dtype=np.float64)
        cpu = lambda k: out[k].cpu().numpy()
        return (self.state_arr, cpu('partial'), cpu('total'), cpu('state_next'), cpu('done'), rwrd_arr, cpu('term'),
                float(out['ep_return'][0]), self.ee_pos_arr)

    # ------------------------------------------------------------------------------ rollouts
    def horizon(self, ICS):
        """NSTEPS_SH = NSTEPS - int(t0 / dt) (RL.py:201): fp64 division, truncation -- evaluated on the host in fp64."""
        ICS = np.asarray(ICS, dtype=np.float64).reshape(-1, self.conf.nb_state)
        return (self.conf.NSTEPS - (ICS[:, -1] / self.conf.dt).astype(np.int64)).astype(np.int32)

    # Rollout engines: 'tc' = tcgen05 fp16-split persistent kernel (cacto_rollout_tc16, default), 'tf32' = tcgen05 3xTF32
    # kernel (cacto_rollout_tc), 'fma' = fp32 CUDA-core kernel (cacto_rollout; also runs the ep = 0 zero-control rollouts).
    rollout_engine = 'tc'
    use_update_graph = True          # learn_and_update replays a captured update (RL.UpdateGraph) instead of launching it eagerly
    use_pipelined_updates = True     # ... and, on one GPU, overlaps consecutive updates (RL.PipelinedUpdateGraph)

    def _rollout_kernel(self, ep, engine=None):
        """The kernel that runs the rollouts of episode ``ep`` on ``engine`` (default: ``rollout_engine``): 'fma' for the
        zero-control rollouts of ep = 0; 'width' (cacto_rollout_width) for an actor whose hidden widths are not 256, whatever
        the engine (the tcgen05 kernels are 256-wide); 'tf32' for 'tc' when the system has more inputs than the fp16 kernel
        holds (UR5: its fp64 dynamics, not the actor, bound the time there, and the 3xTF32 kernel is the faster one,
        profiles/README.md); otherwise the engine itself."""
        engine = engine or self.rollout_engine
        if engine not in ('tc', 'tf32', 'fma'):
            raise ValueError('unknown rollout engine %r' % (engine,))
        if ep == 0:
            return 'fma'
        if self.actor_model.kind == 'actor_width':
            return 'width'
        if engine == 'tc' and self.actor_model.ns > TC16_MAX_NS:
            return 'tf32'
        return engine

    def _launch_rollout(self, ep, ics, hz, T_max, states, controls, flags, rewards, B, engine=None, prepare=True):
        kernel = self._rollout_kernel(ep, engine)
        use_actor = int(ep != 0)
        am = self.actor_model
        if kernel == 'width':
            w1, w2 = am.dims[1], am.dims[2]
            if states.is_cuda:
                ops.rollout_width(self.env._pt, am.params, w1, w2, ics, hz, T_max, states, controls, flags, rewards)
            else:                # zero-copy mode: pinned host outputs through UVA, plain C ABI
                check(lib.cacto_rollout_width(self.env._p, ptr(am.params), w1, w2, ptr(ics), ptr(hz), T_max, ptr(states), ptr(controls), ptr(flags),
                                              ptr(rewards), B, stream_ptr()), 'rollout_width')
        elif kernel == 'tc':
            img = getattr(self, '_w2img16', None)
            if img is None:
                img = torch.empty(int(lib.cacto_actor_tc16_image_bytes()), dtype=torch.uint8, device=am.params.device)
                self._w2img16 = img
            if prepare:          # the W2 image follows the policy version; sub-batches of one call share it
                ops.actor_tc16_prepare(am.params, am.ns, am.na, img)
            if states.is_cuda:
                ops.rollout_tc16(self.env._pt, am.params, img, ics, hz, T_max, states, controls, flags, rewards)
            else:                # zero-copy mode: the outputs are pinned HOST buffers addressed through UVA (no torch CUDA tensor): plain C ABI
                check(lib.cacto_rollout_tc16(self.env._p, ptr(am.params), ptr(img), ptr(ics), ptr(hz), T_max, ptr(states), ptr(controls), ptr(flags),
                                             ptr(rewards), B, stream_ptr()), 'rollout_tc16')
        elif kernel == 'tf32':
            img = getattr(self, '_w2img', None)
            if img is None:
                img = torch.empty(int(lib.cacto_actor_tc_image_floats()), dtype=torch.float32, device=am.params.device)
                self._w2img = img
            if prepare:
                check(lib.cacto_actor_tc_prepare(ptr(am.params), am.ns, am.na, ptr(img), stream_ptr()), 'actor_tc_prepare')
            check(lib.cacto_rollout_tc(self.env._p, ptr(am.params), ptr(img), ptr(ics), ptr(hz), T_max, ptr(states), ptr(controls), ptr(flags),
                                       ptr(rewards), B, stream_ptr()), 'rollout_tc')
        else:
            if states.is_cuda:
                ops.rollout(self.env._pt, am.params if use_actor else None, use_actor, ics, hz, T_max, states, controls, flags, rewards)
            else:
                check(lib.cacto_rollout(self.env._p, ptr(am.params if use_actor else None), use_actor, ptr(ics), ptr(hz), T_max, ptr(states), ptr(controls),
                                        ptr(flags), ptr(rewards), B, stream_ptr()), 'rollout')

    def rollout_batch(self, ICS, ep, horizon=None, with_reward=False, engine=None):
        """All warm-starts of RL.py:197-233 for ICS[B, ns] in one launch of the fused actor+dynamics kernel.
        Returns a dict: states [T_max+1, ns, B] and controls [T_max, na, B] (fp64, structure-of-arrays, time-major;
        ``states.permute(2, 0, 1)`` is the reference's per-rollout [T+1, ns] view), horizon [B] (NSTEPS_SH),
        success [B] (0 where a NaN was met, RL.py:229-231), optionally rewards [T_max+1, B]."""
        c = self.conf
        dev = _device()
        ics = _as_cuda(ICS, torch.float64).reshape(-1, c.nb_state)
        B = ics.shape[0]
        if horizon is None:
            horizon = self.horizon(ics.cpu().numpy() if isinstance(ICS, torch.Tensor) else ICS)
        hz = torch.as_tensor(np.asarray(horizon, dtype=np.int32)).to(dev) if not isinstance(horizon, torch.Tensor) else horizon.to(dev, torch.int32)
        T_max = int(c.NSTEPS)
        states = torch.full((T_max + 1, c.nb_state, B), float('nan'), dtype=torch.float64, device=dev)
        controls = torch.full((T_max, c.nb_action, B), float('nan'), dtype=torch.float64, device=dev)
        flags = torch.empty(B, dtype=torch.int32, device=dev)
        rewards = torch.full((T_max + 1, B), float('nan'), dtype=torch.float64, device=dev) if with_reward else None
        self._launch_rollout(ep, ics, hz, T_max, states, controls, flags, rewards, B, engine)
        self._retry_flagged(ep, ics, hz, T_max, states, controls, flags, rewards, engine)
        out = dict(states=states, controls=controls, horizon=hz, success=flags)
        if with_reward:
            out['rewards'] = rewards
        return out

    def _retry_flagged(self, ep, ics, hz, T_max, states, controls, flags, rewards, engine=None):
        """The fp16-split kernel ('tc') flags a rollout failed when a hidden activation leaves the fp16 range (+-2047
        after scaling, rollout_tc16.cu) -- a limit the reference does not have: RL.py:229-231 aborts on NaN only and trained
        actors are unbounded (SURVEY.md quirk Q11).  Flagged rollouts are therefore rolled out again on the fp32 'fma' engine and
        patched into the outputs; only rollouts that fail there too (a NaN state, as in the reference) stay flagged.
        Costs one device->host read of the failure count per call.  Returns the number of rollouts re-run."""
        if self._rollout_kernel(ep, engine) != 'tc':
            return 0
        bad = (flags == 0).nonzero().reshape(-1)
        n = int(bad.numel())
        if n == 0:
            return 0
        dev = flags.device
        ns, na = states.shape[1], controls.shape[1]
        st = torch.full((T_max + 1, ns, n), float('nan'), dtype=torch.float64, device=dev)
        ct = torch.full((T_max, na, n), float('nan'), dtype=torch.float64, device=dev)
        fl = torch.empty(n, dtype=torch.int32, device=dev)
        rw = torch.full((T_max + 1, n), float('nan'), dtype=torch.float64, device=dev) if rewards is not None else None
        self._launch_rollout(ep, ics[bad].contiguous(), hz[bad].contiguous(), T_max, st, ct, fl, rw, n, 'fma')
        states[:, :, bad] = st
        controls[:, :, bad] = ct
        flags[bad] = fl
        if rewards is not None:
            rewards[:, bad] = rw
        return n

    class _PendingRollouts:
        """Handle of ``rollout_to_host(..., wait=False)``: ``wait()`` blocks until the trajectories are in the host buffers
        (and re-runs rollouts the fp16 engine flagged); ``horizon`` = NSTEPS_SH per rollout."""

        def __init__(self, finish, horizon):
            self._finish, self.horizon = finish, horizon

        def wait(self):
            if self._finish is not None:
                self._finish()
                self._finish = None
            return self.horizon

    def rollout_to_host(self, ics_host, ep, states_host, controls_host, flags_host, mode='pipelined', engine=None, n_chunks=8, wait=True,
                        compact=False):
        """Host-to-host rollouts for the TO feeder: ``ics_host`` [B, ns] fp64 (pinned) -> ``states_host``
        [T_max+1, ns, B], ``controls_host`` [T_max, na, B] fp64 and ``flags_host`` [B] int32 (pinned).
        mode 'pipelined' (default): the batch is rolled out in ``n_chunks`` sub-batches; while sub-batch k + 1 runs, the copy
        engine moves the trajectories of sub-batch k into their columns of the host buffers (strided DMA, ~55 GB/s).
        mode 'zero_copy': the kernel stores straight into the pinned host buffers over PCIe (UVA, ~48 GB/s).
        mode 'staged': H2D, kernel into HBM, D2H.
        ``compact=True`` (pipelined mode): 25 % fewer bytes over PCIe, bit-reconstructible -- ``states_host`` is [T_max+1, ns-1, B] (no
        time row: t_k = t_0 + k dt by repeated addition is what the kernel computes) and ``controls_host`` [T_max, na, B] **float32**
        (the actor's outputs are fp32 values widened to fp64); ``CompactRollouts`` rebuilds the reference's per-rollout arrays.
        ``wait=False`` (pipelined mode): returns a handle right after the work is queued; a caller that alternates between two sets of
        host buffers queues batch k + 1 before waiting for batch k, so that the first kernel and the host-side bookkeeping of a batch
        overlap the tail of the previous batch's copies."""
        c = self.conf
        dev = _device()
        B = ics_host.shape[0]
        T_max = int(c.NSTEPS)
        ns, na = int(c.nb_state), int(c.nb_action)
        ics = ics_host.to(dev, non_blocking=True)
        hz_np = self.horizon(ics_host.numpy())
        hz = torch.as_tensor(hz_np).to(dev, non_blocking=True)
        if compact:
            if mode != 'pipelined':
                raise ValueError("compact transfers are a mode of the 'pipelined' path")
            if tuple(states_host.shape) != (T_max + 1, ns - 1, B) or states_host.dtype != torch.float64 or \
                    tuple(controls_host.shape) != (T_max, na, B) or controls_host.dtype != torch.float32:
                raise ValueError('compact=True: states_host [T+1, ns-1, B] float64 and controls_host [T, na, B] float32 expected')
        if mode == 'pipelined':
            bc = -(-B // max(1, int(n_chunks)))
            bc = -(-bc // 128) * 128                               # whole 128-rollout tiles per sub-batch
            st = getattr(self, '_pipe_stage', None)
            if st is None or st['bc'] != bc:
                st = dict(bc=bc, copy_stream=torch.cuda.Stream(device=dev),
                          s=[torch.empty((T_max + 1) * ns * bc, dtype=torch.float64, device=dev) for _ in range(2)],
                          u=[torch.empty(T_max * na * bc, dtype=torch.float64, device=dev) for _ in range(2)],
                          f=[torch.empty(bc, dtype=torch.int32, device=dev) for _ in range(2)])
                self._pipe_stage = st
            main, side = torch.cuda.current_stream(), st['copy_stream']
            copied = st.setdefault('copied', [None, None])         # (kept across calls: the staging slots are shared by batches in flight)
            for k, b0 in enumerate(range(0, B, bc)):
                n = min(bc, B - b0)
                slot = k & 1
                if copied[slot] is not None:
                    main.wait_event(copied[slot])                  # the copy of the sub-batch that used this staging slot is done
                sk = st['s'][slot][:(T_max + 1) * ns * n].view(T_max + 1, ns, n)
                uk = st['u'][slot][:T_max * na * n].view(T_max, na, n)
                fk = st['f'][slot][:n]
                self._launch_rollout(ep, ics[b0:b0 + n], hz[b0:b0 + n], T_max, sk, uk, fk, None, n, engine, prepare=(k == 0))
                if compact:                                        # narrow the controls (exact); the copy itself skips the time rows
                    if 'uc' not in st:
                        st['uc'] = [torch.empty(T_max * na * bc, dtype=torch.float32, device=dev) for _ in range(2)]
                    uc = st['uc'][slot][:T_max * na * n]
                    check(lib.cacto_narrow_f64_to_f32(ptr(uk), ptr(uc), T_max * na * n, main.cuda_stream), 'narrow')
                done = torch.cuda.Event()
                done.record(main)
                side.wait_event(done)
                sp = side.cuda_stream
                if compact:
                    check(lib.cacto_copy3d_to_host(states_host.data_ptr() + 8 * b0, 8 * B, ns - 1, ptr(sk), 8 * n, ns, 8 * n, ns - 1, T_max + 1, sp),
                          'copy3d')
                    check(lib.cacto_copy2d_to_host(controls_host.data_ptr() + 4 * b0, 4 * B, ptr(uc), 4 * n, 4 * n, T_max * na, sp), 'copy2d')
                else:
                    check(lib.cacto_copy2d_to_host(states_host.data_ptr() + 8 * b0, 8 * B, ptr(sk), 8 * n, 8 * n, (T_max + 1) * ns, sp), 'copy2d')
                    check(lib.cacto_copy2d_to_host(controls_host.data_ptr() + 8 * b0, 8 * B, ptr(uk), 8 * n, 8 * n, T_max * na, sp), 'copy2d')
                check(lib.cacto_copy2d_to_host(flags_host.data_ptr() + 4 * b0, 4 * n, ptr(fk), 4 * n, 4 * n, 1, sp), 'copy2d')
                copied[slot] = torch.cuda.Event()
                copied[slot].record(side)
            if not wait:
                tail = torch.cuda.Event()
                tail.record(side)

                def finish():
                    tail.synchronize()
                    self._patch_flagged_host(ics_host, hz_np, ep, states_host, controls_host, flags_host, engine)
                return self._PendingRollouts(finish, hz_np)
            side.synchronize()
        elif mode == 'zero_copy':
            flags = torch.empty(B, dtype=torch.int32, device=dev)
            self._launch_rollout(ep, ics, hz, T_max, states_host, controls_host, flags, None, B, engine)
            flags_host.copy_(flags, non_blocking=True)
        else:
            buf = getattr(self, '_host_stage', None)
            if buf is None or buf[0].shape[2] != B:
                buf = (torch.empty((T_max + 1, c.nb_state, B), dtype=torch.float64, device=dev),
                       torch.empty((T_max, c.nb_action, B), dtype=torch.float64, device=dev),
                       torch.empty(B, dtype=torch.int32, device=dev))
                self._host_stage = buf
            self._launch_rollout(ep, ics, hz, T_max, buf[0], buf[1], buf[2], None, B, engine)
            states_host.copy_(buf[0], non_blocking=True)
            controls_host.copy_(buf[1], non_blocking=True)
            flags_host.copy_(buf[2], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        self._patch_flagged_host(ics_host, hz_np, ep, states_host, controls_host, flags_host, engine)
        return hz_np if wait else self._PendingRollouts(None, hz_np)

    def _patch_flagged_host(self, ics_host, hz_np, ep, states_host, controls_host, flags_host, engine):
        """fp16-range failures of the 'tc' kernel (see _retry_flagged): re-run on 'fma' and patch the host buffers."""
        if self._rollout_kernel(ep, engine) == 'tc':
            bad = (flags_host == 0).nonzero().reshape(-1)
            if bad.numel() > 0:
                r = self.rollout_batch(ics_host[bad], ep, horizon=hz_np[bad.numpy()], engine='fma')
                nrow = states_host.shape[1]                        # ns, or ns - 1 for compact transfers
                states_host[:, :, bad] = r['states'][:, :nrow, :].cpu()
                controls_host[:, :, bad] = r['controls'].cpu().to(controls_host.dtype)
                flags_host[bad] = r['success'].cpu()

    def create_TO_init(self, ep, ICS):
        """RL.py:197-233 for one initial condition -> (ICS, init_TO_states[T+1, ns], init_TO_controls[T, na], T, success)."""
        self.init_rand_state = ICS
        self.NSTEPS_SH = int(self.horizon(ICS)[0])
        if self.NSTEPS_SH == 0:
            return None, None, None, None, 0
        T = self.NSTEPS_SH
        r = self.rollout_batch(np.asarray(ICS, dtype=np.float64).reshape(1, -1), ep)
        if int(r['success'][0]) == 0:
            return None, None, None, None, 0
        init_TO_states = r['states'][:T + 1, :, 0].cpu().numpy()
        init_TO_controls = r['controls'][:T, :, 0].cpu().numpy()
        self.control_arr = np.empty((T, self.conf.nb_action))
        self.state_arr = np.empty((T + 1, self.conf.nb_state))
        self.ee_pos_arr = np.empty((T + 1, 3))
        self.state_arr[0, :] = ICS
        self.ee_pos_arr[0, :] = self.env.get_end_effector_position(self.state_arr[0, :])
        return self.init_rand_state, init_TO_states, init_TO_controls, self.NSTEPS_SH, 1


class UpdateGraph:
    """One critic+actor update (RL.py:101-118) as a replayable CUDA graph: 6 kernel nodes
    (schedule, critic gradient, critic Adam + Polyak, schedule, actor gradient, actor Adam), plus the NCCL
    all-reduces when data-parallel.  At the reference's batch sizes (64/128) the update is launch-latency bound;
    replaying a graph removes the per-launch host cost."""

    def __init__(self, rl, B):
        self.rl, self.B = rl, B
        c = rl.conf
        dev = _device()
        ns = c.nb_state
        f32 = dict(dtype=torch.float32, device=dev)
        self.io = dict(state=torch.zeros((B, ns), **f32), state_next=torch.zeros((B, ns), **f32), partial_rtg=torch.zeros((B, 1), **f32),
                       dVdx=torch.zeros((B, ns), **f32), done=torch.zeros((B, 1), **f32), term=torch.zeros((B, 1), dtype=torch.float64, device=dev),
                       weights=torch.ones((B, 1), **f32), rtg=torch.zeros((B, 1), **f32), V=torch.zeros((B, 1), **f32),
                       V_target=torch.zeros((B, 1), **f32))
        nets = (rl.actor_model, rl.critic_model, rl.target_critic)
        opts = (rl.critic_optimizer, rl.actor_optimizer)
        for o, n in ((rl.critic_optimizer, rl.critic_model), (rl.actor_optimizer, rl.actor_model)):
            o.moments(n)
            o._device_state(dev)
        # In peer mode the gradient blocks are mapped by the other ranks, whose k_adam_peer of the previous eager update may still be
        # summing them: nothing may clear them before every rank's stream has drained (update.cu: "a rank never clears its own block").
        self._quiesce()
        for n in nets:
            n.grad.zero_()
        self._quiesce()
        # snapshot the training state, warm up on a side stream (lazy initialisation), capture, restore
        snap = [(t, t.clone()) for n in nets for t in (n.params, n.params_T) if t is not None]
        snap += [(t, t.clone()) for o in opts for st in o._state.values() for t in st]
        snap += [(o._dev['step'], o._dev['step'].clone()) for o in opts]
        its = [o.iterations for o in opts]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                rl._update_static(self.io)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            rl._update_static(self.io)
        for t, old in snap:
            t.copy_(old)
        for o, it in zip(opts, its):
            o.iterations = it
        self._quiesce()
        for n in nets:
            n.grad.zero_()
        self._quiesce()

    def _quiesce(self):
        """All launches of this rank done and -- data-parallel -- of every other rank too."""
        torch.cuda.synchronize()
        if self.rl._peer is not None and getattr(self.rl.dist, 'barrier', None) is not None:
            self.rl.dist.barrier()
            torch.cuda.synchronize()

    def replay(self):
        self.graph.replay()
        self.rl.critic_optimizer.iterations += 1
        self.rl.actor_optimizer.iterations += 1
        return self.io['rtg'], self.io['V'], self.io['V_target']


class PipelinedUpdateGraph:
    """Consecutive updates of RL_AC.update (RL.py:101-111) software-pipelined on one GPU.

    ``compute_critic_grad`` never evaluates the actor (NeuralNetwork.py:150-178) and the actor step of update i only needs the critic
    as update i left it (RL.py:104-109), so the actor step of update i and the critic GRADIENT of update i + 1 are independent: replay
    i + 1 runs them side by side (two branches of one CUDA graph) and applies the critic's Adam step only once the actor gradient of
    update i has read the critic.  Every kernel sees exactly the inputs it sees in the sequential order, so the weights after
    ``flush()`` are those of the sequential updates; at the conf batches, where both gradient kernels are latency-bound chains on
    32 of the 148 SMs, the period drops from the sum of the two chains to the longer one.

    Use: ``buffer.sample(out=g.io)`` -> ``rtg, V, V_target = g.replay()`` -> ... -> ``g.flush()`` before the actor is read (rollouts,
    checkpoints).  Two sets of input tensors alternate (``g.io`` is the set the next ``replay`` trains the critic on)."""

    def __init__(self, rl, B):
        self.rl, self.B = rl, B
        c, nn = rl.conf, rl.NN
        world = rl.dist.get_world_size() if rl.dist is not None else 1
        if world != 1:
            raise ValueError('PipelinedUpdateGraph is single-GPU: the peer-memory exchange assumes alternating critic / actor steps')
        if rl.critic_model.kind != 'critic_sine' or nn._use_tc(B):
            raise ValueError("PipelinedUpdateGraph needs the fused 'sine' engine (the tcgen05 engine shares one workspace between the two steps)")
        dev = _device()
        ns = c.nb_state
        f32 = dict(dtype=torch.float32, device=dev)

        def make_io():
            return dict(state=torch.zeros((B, ns), **f32), state_next=torch.zeros((B, ns), **f32), partial_rtg=torch.zeros((B, 1), **f32),
                        dVdx=torch.zeros((B, ns), **f32), done=torch.zeros((B, 1), **f32), term=torch.zeros((B, 1), dtype=torch.float64, device=dev),
                        weights=torch.ones((B, 1), **f32), rtg=torch.zeros((B, 1), **f32), V=torch.zeros((B, 1), **f32),
                        V_target=torch.zeros((B, 1), **f32))
        self.ios = (make_io(), make_io())
        self.turn, self.pending = 0, None
        nets = (rl.actor_model, rl.critic_model, rl.target_critic)
        opts = (rl.critic_optimizer, rl.actor_optimizer)
        for o, n in ((rl.critic_optimizer, rl.critic_model), (rl.actor_optimizer, rl.actor_model)):
            o.moments(n)
            o._device_state(dev)
        torch.cuda.synchronize()
        for n in nets:
            n.grad.zero_()
        # snapshot the training state, warm up on a side stream (lazy initialisation), capture, restore
        snap = [(t, t.clone()) for n in nets for t in (n.params, n.params_T) if t is not None]
        snap += [(t, t.clone()) for o in opts for st in o._state.values() for t in st]
        snap += [(o._dev['step'], o._dev['step'].clone()) for o in opts]
        its = [o.iterations for o in opts]
        self._side = torch.cuda.Stream()
        warm = torch.cuda.Stream()
        warm.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(warm):
            for io in self.ios:
                rl._critic_step_static(io)
                rl._actor_step_static(io)
        torch.cuda.current_stream().wait_stream(warm)
        torch.cuda.synchronize()

        def capture(fn):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                fn()
            return g
        self.critic_only = [capture(lambda io=io: rl._critic_step_static(io)) for io in self.ios]
        self.actor_only = [capture(lambda io=io: rl._actor_step_static(io)) for io in self.ios]
        self.steady = [capture(lambda p=p: self._steady(p)) for p in (0, 1)]
        for t, old in snap:
            t.copy_(old)
        for o, it in zip(opts, its):
            o.iterations = it
        torch.cuda.synchronize()
        for n in nets:
            n.grad.zero_()
        torch.cuda.synchronize()

    def _steady(self, p):
        """Critic step on ios[p] beside the actor step on ios[1 - p] (the previous batch); both schedules in one launch."""
        rl, nn = self.rl, self.rl.NN
        c = rl.conf
        io_c, io_a = self.ios[p], self.ios[1 - p]
        B = self.B
        cm, tc, am = rl.critic_model, rl.target_critic, rl.actor_model
        main, side = torch.cuda.current_stream(), self._side
        type(rl.critic_optimizer).prepare_pair(rl.critic_optimizer, rl.actor_optimizer, cm.params.device, zero=nn.last_critic_loss)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            nn.launch_actor_grad(am, cm, io_a['state'], io_a['term'], 1.0 / float(B), None, B)
            read = torch.cuda.Event()
            read.record(side)                                    # the previous critic has been read: its Adam step may go ahead
            rl._reduce_and_step(rl.actor_optimizer, am, cm, prepared=True)
        nn.launch_critic_grad(cm, tc, io_c['state'], io_c['state_next'], io_c['partial_rtg'], io_c['dVdx'], io_c['done'], io_c['weights'],
                              1.0 / float(B), io_c['rtg'], io_c['V'], io_c['V_target'], B)
        main.wait_event(read)
        if c.MC:
            rl._reduce_and_step(rl.critic_optimizer, cm, am, prepared=True)
        else:
            rl._reduce_and_step(rl.critic_optimizer, cm, am, target=tc, tau=c.UPDATE_RATE, prepared=True)
        main.wait_stream(side)

    @property
    def io(self):
        return self.ios[self.turn]

    def replay(self):
        """Critic step on the batch in ``io`` (and the outstanding actor step of the previous batch); returns that batch's
        (rtg, V, V_target) tensors, valid until the replay after next."""
        p = self.turn
        if self.pending is None:
            self.critic_only[p].replay()
        else:
            self.steady[p].replay()
            self.rl.actor_optimizer.iterations += 1
        self.rl.critic_optimizer.iterations += 1
        self.pending, self.turn = p, 1 - p
        io = self.ios[p]
        return io['rtg'], io['V'], io['V_target']

    def flush(self):
        """Run the outstanding actor step: afterwards actor, critic and target are those of the sequential updates."""
        if self.pending is not None:
            self.actor_only[self.pending].replay()
            self.rl.actor_optimizer.iterations += 1
            self.pending = None
