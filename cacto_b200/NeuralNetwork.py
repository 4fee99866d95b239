"""Host-side mirror of the reference's ``NeuralNetwork.py`` (class ``NN``) on the CUDA kernels.

Networks are flat float32 parameter blocks in HBM in Keras order [W1 (in x out), b1, W2, b2, ...]
(include/cacto_b200.h), wrapped by ``Network`` which offers the slice of the Keras model surface the
reference uses: ``trainable_variables`` / ``variables``, ``get_weights`` / ``set_weights``,
``save_weights`` / ``load_weights`` and ``__call__``.

  NN.eval                 -> cacto_actor_forward / cacto_critic_forward   (NeuralNetwork.py:130-138)
  NN.compute_critic_grad  -> cacto_critic_grad                            (NeuralNetwork.py:150-178)
  NN.compute_actor_grad   -> cacto_actor_grad                             (NeuralNetwork.py:180-232)

``NN(..., deterministic=True)`` runs the 'sine' critic and actor gradients through the ``*_grad_det`` / ``*_grad_tc_det`` entry points:
the same kernels of both update engines with every cross-CTA and cross-warp sum taken in a fixed order (include/cacto_b200.h), so
that an update repeated on the same inputs gives the same bits.

An actor whose hidden widths (conf.NH1, conf.NH2) are not 256 is an ``'actor_width'`` network: the same Keras layout and layer
names, no transposed copy, run by the width-generic kernels of csrc/actor_width.cu (cacto_rollout_width / cacto_actor_forward_width /
cacto_actor_grad_width) with the widths passed at run time.

The regularisers the reference attaches to its layers are inert there (gradients are taken of the loss
only, ``model.losses`` is never added: SURVEY.md quirk Q6) and are therefore not represented.
The default critic ('sine', every conf) runs on the fused tiled kernels of csrc/update.cu; the elu / relu / sine-elu
variants (NeuralNetwork.py:65-93,110-128) run on the generic one-CTA-per-sample kernels of csrc/mlp_generic.cu
(``Network.kind == 'critic_generic'``), with the same methods and return values.
"""
import math
import weakref

import numpy as np
import torch

from . import _lib
from ._lib import check, lib, ptr, stream_ptr
from .environment import _as_cuda, _device
from .ops import ops

CRITIC_HIDDEN = (64, 64, 128, 128)
ACTOR_MAX_WIDTH = 512        # CACTO_ACTOR_MAX_WIDTH (include/cacto_b200.h)
GENERIC_MAX_WIDTH = 256      # units per layer of the generic critic kernels (csrc/mlp_generic.cu)


class Network:
    """A dense network stored as one flat float32 block (+ its per-layer transposed copy and a gradient
    accumulator).  kind: 'actor' (LeakyReLU 0.3, hidden widths 256), 'actor_width' (the same at any hidden widths 1..512, no
    transposed copy), 'critic_sine', or 'critic_generic' (any layer table, ``acts`` per layer: 'sin' | 'elu' | 'leaky' | 'linear';
    no transposed copy)."""

    _registry = weakref.WeakValueDictionary()      # params address -> Network (apply_gradients looks the owner up); weak: GPU blocks are freed with the net

    def __init__(self, kind, ns, na, dims, acts=None):
        self.kind, self.ns, self.na, self.dims = kind, int(ns), int(na), list(dims)
        self.n = sum(i * o + o for i, o in zip(dims[:-1], dims[1:]))
        if acts is None:
            acts = (['leaky'] * (len(dims) - 2) if self.is_actor else ['sin'] * (len(dims) - 2)) + ['linear']
        self.acts = list(acts)
        self.desc = _lib.make_mlp_desc(self.dims, self.acts)
        dev = _device()
        self.params = torch.zeros(self.n, dtype=torch.float32, device=dev)
        if kind == 'actor_width':
            assert len(self.dims) == 4 and self.n == lib.cacto_actor_width_param_count(self.ns, self.na, self.dims[1], self.dims[2]), self.dims
            self.params_T = None
        elif kind == 'critic_generic':
            self.params_T = None
        else:
            expect = lib.cacto_critic_param_count(self.ns) if kind == 'critic_sine' else lib.cacto_actor_param_count(self.ns, self.na)
            assert self.n == expect, (self.n, expect)
            self.params_T = torch.zeros(self.n, dtype=torch.float32, device=dev)
        self.grad = torch.zeros(self.n, dtype=torch.float32, device=dev)
        self._views = self._make_views(self.params)
        self._grad_views = self._make_views(self.grad)
        Network._registry[self.params.data_ptr()] = self

    @property
    def is_actor(self):
        return self.kind in ('actor', 'actor_width')

    @property
    def is_critic(self):
        return int(self.kind == 'critic_sine')

    def _make_views(self, flat):
        out, o = [], 0
        for i, k in zip(self.dims[:-1], self.dims[1:]):
            out.append(flat[o:o + i * k].view(i, k))
            o += i * k
            out.append(flat[o:o + k])
            o += k
        return out

    # -- Keras-like surface -------------------------------------------------------------------
    @property
    def trainable_variables(self):
        return self._views

    variables = trainable_variables

    def get_weights(self):
        return [v.detach().cpu().numpy().copy() for v in self._views]

    def set_weights(self, weights):
        assert len(weights) == len(self._views)
        for v, w in zip(self._views, weights):
            w = torch.as_tensor(np.asarray(w, dtype=np.float32))
            assert tuple(w.shape) == tuple(v.shape), (tuple(w.shape), tuple(v.shape))
            v.copy_(w)
        self.refresh_transposed()

    def refresh_transposed(self):
        if self.params_T is None:
            return
        ops.transpose_params(self.params, self.params_T, self.is_critic, self.ns, self.na)

    def _keras_layer_names(self):
        """Layer names of the reference's Keras models with weights, in topological order (as in its archived .h5 files)."""
        L = len(self.dims) - 1
        if self.is_actor:
            return ['dense' if l == 0 else f'dense_{l}' for l in range(L)]
        if self.kind == 'critic_sine':
            return ['sinusodial_representation_dense' if l == 0 else f'sinusodial_representation_dense_{l}' for l in range(L - 1)] + ['dense_3']
        return [f'dense_{l}' for l in range(L)]

    def save_weights(self, path):
        """``<path>.h5``: a Keras-2.11 ``save_weights`` HDF5 file as the reference writes it (RL.py:191-195; h5weights.save_keras_weights);
        any other path: ``.npz``."""
        path = str(path)
        if path.endswith('.h5'):
            from .h5weights import save_keras_weights
            save_keras_weights(path, self.get_weights(), self._keras_layer_names())
            return
        np.savez(path if path.endswith('.npz') else path + '.npz', *self.get_weights())

    def load_weights(self, path):
        """A Keras ``.h5`` file written by the reference or by save_weights (RL.py:91-97,191-195), or an ``.npz``."""
        import os
        path = str(path)
        if path.endswith('.h5') and not os.path.exists(path) and os.path.exists(path[:-3] + '.npz'):
            path = path[:-3] + '.npz'
        if path.endswith('.h5'):
            from .h5weights import load_keras_weights, load_keras_weights_by_tree
            try:
                w = load_keras_weights_by_tree(path)         # Keras' own rule: the order of the layer_names attribute
                if len(w) != len(self._views):
                    raise ValueError
            except Exception:
                w = load_keras_weights(path, self.ns)        # layout-agnostic reader: chains the layers by shape
            self.set_weights(w)
            return
        z = np.load(path if path.endswith('.npz') else path + '.npz')
        self.set_weights([z[f'arr_{i}'] for i in range(len(self._views))])

    def __call__(self, x, training=True):
        raise TypeError('call NN.eval(network, input): normalisation is fused into the forward kernel')


def _glorot(rng, i, o):
    lim = math.sqrt(6.0 / (i + o))
    return rng.uniform(-lim, lim, (i, o)).astype(np.float32)


class NN:
    """NeuralNetwork.py:10-232."""

    def __init__(self, env, conf, w_S=0, seed=None, deterministic=False):
        """``deterministic``: bit-reproducible gradients (fixed-order sums instead of fp32 atomics) for the 'sine' critic and its
        actor.  For a fixed GPU model, build, system, batch size and world size the same inputs then give the same bits in every
        gradient, weight, Adam moment, rtg, V, V_target and ``last_critic_loss``.  The generic critic variants have no such path."""
        self.env = env
        self.conf = conf
        self.w_S = w_S
        self.deterministic = bool(deterministic)
        if self.deterministic and getattr(conf, 'critic_type', 'sine') != 'sine':
            raise ValueError(f"deterministic=True needs critic_type 'sine' (got {conf.critic_type!r}): the generic critic kernels sum "
                             'their gradients with one atomic per weight and sample')
        self._rng = np.random.default_rng(seed)
        self._p = env._p
        self._pt = env._pt
        self.last_critic_loss = torch.zeros(1, dtype=torch.float32, device=_device())

    # -- model constructors ---------------------------------------------------------------------
    def create_actor(self):
        """NeuralNetwork.py:51-63: Dense(NH1) LeakyReLU Dense(NH2) LeakyReLU Dense(na); glorot-uniform kernels, zero biases.
        NH1 = NH2 = 256 (every reference conf) runs on the fused kernels ('actor'); any other widths in 1..512 on the width-generic
        ones ('actor_width')."""
        c = self.conf
        nh1, nh2 = int(c.NH1), int(c.NH2)
        if not (1 <= nh1 <= ACTOR_MAX_WIDTH and 1 <= nh2 <= ACTOR_MAX_WIDTH):
            raise ValueError(f'actor hidden widths NH1 = {nh1}, NH2 = {nh2}: each must be in 1..{ACTOR_MAX_WIDTH}')
        kind = 'actor' if (nh1, nh2) == (256, 256) else 'actor_width'
        net = Network(kind, c.nb_state, c.nb_action, [c.nb_state, nh1, nh2, c.nb_action])
        w = []
        for i, o in zip(net.dims[:-1], net.dims[1:]):
            w += [_glorot(self._rng, i, o), np.zeros(o, np.float32)]
        net.set_weights(w)
        return net

    def create_critic_sine(self):
        """NeuralNetwork.py:95-108: four SIREN layers (64, 64, 128, 128; tf_siren w0 = 1: kernel U(+-sqrt(6/fan_in)),
        bias he_uniform U(+-sqrt(6/units))) and a linear Dense(1)."""
        c = self.conf
        net = Network('critic_sine', c.nb_state, c.nb_action, [c.nb_state] + list(CRITIC_HIDDEN) + [1])
        w = []
        for i, o in zip(net.dims[:-2], net.dims[1:-1]):
            lk, lb = math.sqrt(6.0 / i), math.sqrt(6.0 / o)
            w += [self._rng.uniform(-lk, lk, (i, o)).astype(np.float32), self._rng.uniform(-lb, lb, o).astype(np.float32)]
        w += [_glorot(self._rng, net.dims[-2], 1), np.zeros(1, np.float32)]
        net.set_weights(w)
        return net

    def _generic_critic(self, hidden, acts, siren):
        """Dense stack ns -> hidden... -> 1 on the generic kernels.  Keras default initialisers (glorot-uniform kernel, zero
        bias) except for the tf_siren layers (kernel U(+-sqrt(6/fan_in)), bias he_uniform), as in create_critic_sine."""
        c = self.conf
        net = Network('critic_generic', c.nb_state, c.nb_action, [c.nb_state] + list(hidden) + [1], list(acts) + ['linear'])
        w = []
        for l, (i, o) in enumerate(zip(net.dims[:-1], net.dims[1:])):
            if l < len(hidden) and siren[l]:
                lk, lb = math.sqrt(6.0 / i), math.sqrt(6.0 / o)
                w += [self._rng.uniform(-lk, lk, (i, o)).astype(np.float32), self._rng.uniform(-lb, lb, o).astype(np.float32)]
            else:
                w += [_glorot(self._rng, i, o), np.zeros(o, np.float32)]
        net.set_weights(w)
        return net

    def create_critic_elu(self):
        """NeuralNetwork.py:65-78: Dense 16, 32, 256, 256 with elu, Dense(1)."""
        return self._generic_critic((16, 32, 256, 256), ['elu'] * 4, [False] * 4)

    def create_critic_sine_elu(self):
        """NeuralNetwork.py:80-93: SIREN(64), Dense(64, elu), SIREN(128), Dense(128, elu), Dense(1)."""
        return self._generic_critic((64, 64, 128, 128), ['sin', 'elu', 'sin', 'elu'], [True, False, True, False])

    def create_critic_relu(self):
        """NeuralNetwork.py:110-128: Dense 16, 32, NH1, NH2 each followed by LeakyReLU() (alpha 0.3), Dense(1); the
        regularisers are inert (quirks Q6, Q14)."""
        c = self.conf
        if max(int(c.NH1), int(c.NH2)) > GENERIC_MAX_WIDTH:
            raise ValueError(f"the 'relu' critic uses NH1 = {c.NH1}, NH2 = {c.NH2} as its widths; the generic critic kernels support at most "
                             f'{GENERIC_MAX_WIDTH} units per layer')
        return self._generic_critic((16, 32, c.NH1, c.NH2), ['leaky'] * 4, [False] * 4)

    # -- forward ------------------------------------------------------------------------------
    def eval(self, NN, input):
        """NeuralNetwork.py:130-138: normalise (utils.py:17-24) + forward.  -> [B, na] or [B, 1] float32."""
        x = _as_cuda(input, torch.float32)
        if x.dim() == 1:
            x = x.reshape(1, -1)
        B = x.shape[0]
        if NN.kind == 'actor':
            out = torch.empty((B, NN.na), dtype=torch.float32, device=x.device)
            ops.actor_forward(self._pt, NN.params, x, out)
        elif NN.kind == 'actor_width':
            out = torch.empty((B, NN.na), dtype=torch.float32, device=x.device)
            ops.actor_forward_width(self._pt, NN.params, NN.dims[1], NN.dims[2], x, out)
        elif NN.kind == 'critic_generic':
            out = torch.empty((B, 1), dtype=torch.float32, device=x.device)
            check(lib.cacto_mlp_forward_generic(self._p, _lib.C.byref(NN.desc), ptr(NN.params), ptr(x), ptr(out), ptr(None), B, stream_ptr()),
                  'mlp_forward_generic')
        else:
            out = torch.empty((B, 1), dtype=torch.float32, device=x.device)
            ops.critic_forward(self._pt, NN.params, x, out, None)
        return out

    def eval_with_gradient(self, critic, input):
        """(V, dV/ds) with dV/ds taken w.r.t. the RAW state as the reference's tapes do (NeuralNetwork.py:162-165,190-195)."""
        x = _as_cuda(input, torch.float32)
        B = x.shape[0]
        V = torch.empty((B, 1), dtype=torch.float32, device=x.device)
        dV = torch.empty((B, critic.ns), dtype=torch.float32, device=x.device)
        if critic.kind == 'critic_generic':
            check(lib.cacto_mlp_forward_generic(self._p, _lib.C.byref(critic.desc), ptr(critic.params), ptr(x), ptr(V), ptr(dV), B, stream_ptr()),
                  'mlp_forward_generic')
        else:
            ops.critic_forward(self._pt, critic.params, x, V, dV)
        return V, dV

    # -- gradient launches (shared by the eager methods below and by RL_AC's CUDA-graph update) -----------
    # Batch size from which the 'sine' critic / actor gradients run on the tensor-core kernels (csrc/update_tc.cu: 128-sample
    # tiles, one tile per SM) instead of the fused fp32-FMA tile kernels (csrc/update.cu).  ``update_engine``: 'auto' | 'fma' | 'tc'.
    # Crossover measured as graph-replayed updates (profiles/README.md): the FMA engine's 16-row tiles fill one wave of the 148 SMs up to
    # 2368 samples (190 us at 2048 vs 197 us on tensor cores) and need a second one beyond (245 vs 204 us at 2560).
    TC_MIN_BATCH = 2400
    update_engine = 'auto'

    def _use_tc(self, B):
        eng = self.update_engine
        if eng not in ('auto', 'fma', 'tc'):
            raise ValueError('unknown update engine %r' % (eng,))
        return eng == 'tc' or (eng == 'auto' and B >= self.TC_MIN_BATCH)

    # partials workspace of the deterministic gradients: one per network and engine (the pipelined update runs the critic and actor
    # gradients concurrently), sized for the batch (ops.det_partials_floats stops growing above CACTO_DET_MAX_SLICES tiles).  A
    # workspace that is outgrown is kept, not freed: a CUDA graph captured with it (RL.UpdateGraph) still writes to it on replay.
    DET_CRITIC, DET_ACTOR, DET_ACTOR_WIDTH, DET_CRITIC_TC, DET_ACTOR_TC = 0, 1, 2, 3, 4

    def _det_partials(self, net, B, nh1=0, nh2=0):
        need = int(ops.det_partials_floats(net, B, self.conf.nb_state, self.conf.nb_action, nh1, nh2))
        cache = self.__dict__.setdefault('_det_ws', {})
        ws = cache.get(net)
        if ws is None or ws.numel() < need:
            if ws is not None:
                self.__dict__.setdefault('_det_ws_outgrown', []).append(ws)
            ws = cache[net] = torch.empty(need, dtype=torch.float32, device=_device())
        return ws

    def _tc_workspace(self, B):
        need = int(ops.update_tc_workspace_bytes(B, self.conf.nb_state, self.conf.nb_action))
        ws = getattr(self, '_tc_ws', None)
        if ws is None or ws.numel() < need:
            ws = torch.empty(need, dtype=torch.uint8, device=_device())       # cudaMalloc: 256-byte aligned or better; checked by the callee
            self._tc_ws = ws
        return ws

    def launch_critic_grad(self, cm, tc, s, sn, pr, dv, d, w, inv_B, rtg, V, Vt, B):
        if cm.kind == 'critic_sine' and self._use_tc(B) and self.deterministic:
            ops.critic_grad_tc_det(self._pt, cm.params, tc.params, float(self.w_S), int(bool(self.conf.MC)), s, sn, pr, dv, d, w, inv_B, cm.grad, rtg, V, Vt,
                                   self.last_critic_loss, self._tc_workspace(B), self._det_partials(self.DET_CRITIC_TC, B))
            return
        if cm.kind == 'critic_sine' and self._use_tc(B):
            ws = self._tc_workspace(B)
            ops.critic_grad_tc(self._pt, cm.params, tc.params, float(self.w_S), int(bool(self.conf.MC)), s, sn, pr, dv, d, w, inv_B, cm.grad, rtg, V, Vt,
                               self.last_critic_loss, ws)
            return
        if cm.kind == 'critic_generic':
            check(lib.cacto_critic_grad_generic(self._p, _lib.C.byref(cm.desc), ptr(cm.params), ptr(tc.params), float(self.w_S),
                                                int(bool(self.conf.MC)), ptr(s), ptr(sn), ptr(pr), ptr(dv), ptr(d), ptr(w), inv_B, ptr(cm.grad),
                                                ptr(rtg), ptr(V), ptr(Vt), ptr(self.last_critic_loss), B, stream_ptr()), 'critic_grad_generic')
        elif self.deterministic:
            ops.critic_grad_det(self._pt, cm.params, cm.params_T, tc.params, float(self.w_S), int(bool(self.conf.MC)), s, sn, pr, dv, d, w, inv_B, cm.grad, rtg,
                                V, Vt, self.last_critic_loss, self._det_partials(self.DET_CRITIC, B))
        else:
            ops.critic_grad(self._pt, cm.params, cm.params_T, tc.params, float(self.w_S), int(bool(self.conf.MC)), s, sn, pr, dv, d, w, inv_B, cm.grad, rtg, V, Vt,
                            self.last_critic_loss)

    def launch_actor_grad(self, am, cm, s, term, inv_B, actions, B):
        if am.kind == 'actor_width' and cm.kind == 'critic_sine' and self.deterministic:
            ops.actor_grad_width_det(self._pt, am.params, am.dims[1], am.dims[2], cm.params, cm.params_T, s, term, inv_B, am.grad, actions,
                                     self._det_partials(self.DET_ACTOR_WIDTH, B, am.dims[1], am.dims[2]))
            return
        if am.kind == 'actor_width' and cm.kind == 'critic_sine':      # whatever the batch size: the tcgen05 engine is 256-wide only
            ops.actor_grad_width(self._pt, am.params, am.dims[1], am.dims[2], cm.params, cm.params_T, s, term, inv_B, am.grad, actions)
            return
        if cm.kind == 'critic_sine' and self._use_tc(B) and self.deterministic:
            ops.actor_grad_tc_det(self._pt, am.params, cm.params, s, term, inv_B, am.grad, actions, self._tc_workspace(B),
                                  self._det_partials(self.DET_ACTOR_TC, B))
            return
        if cm.kind == 'critic_sine' and self._use_tc(B):
            ws = self._tc_workspace(B)
            ops.actor_grad_tc(self._pt, am.params, cm.params, s, term, inv_B, am.grad, actions, ws)
            return
        if cm.kind == 'critic_generic':
            # environment terms from the batched kernels of the reference-facing API (NeuralNetwork.py:185-204), network part generic
            act = self.eval(am, s)
            s_next = self.env.simulate_batch(s, act)
            Fu = self.env.derivative_batch(s, act)
            if getattr(self, '_w_rt', None) is None:
                c = self.conf
                self._w_rt = (torch.zeros(8, dtype=torch.float64, device=s.device), torch.zeros(8, dtype=torch.float64, device=s.device))
                wr, wt = np.zeros(8), np.zeros(8)
                wr[:len(c.cost_weights_running)] = c.cost_weights_running
                wt[:len(c.cost_weights_terminal)] = c.cost_weights_terminal
                self._w_rt[0].copy_(torch.as_tensor(wr)); self._w_rt[1].copy_(torch.as_tensor(wt))
            tm = term.reshape(-1, 1)
            w8 = tm * self._w_rt[1][None, :] + (1.0 - tm) * self._w_rt[0][None, :]                 # NeuralNetwork.py:201
            dr_da = self.env.reward_batch_da(w8, s, act)
            if actions is not None:
                actions.copy_(act)
            check(lib.cacto_actor_grad_generic(self._p, _lib.C.byref(am.desc), ptr(am.params), _lib.C.byref(cm.desc), ptr(cm.params), ptr(s),
                                               ptr(s_next), ptr(Fu), ptr(dr_da), inv_B, ptr(am.grad), B, stream_ptr()), 'actor_grad_generic')
        elif self.deterministic:
            ops.actor_grad_det(self._pt, am.params, am.params_T, cm.params, cm.params_T, s, term, inv_B, am.grad, actions,
                               self._det_partials(self.DET_ACTOR, B))
        else:
            ops.actor_grad(self._pt, am.params, am.params_T, cm.params, cm.params_T, s, term, inv_B, am.grad, actions)

    def custom_logarithm(self, input):
        """NeuralNetwork.py:140-148."""
        x = torch.as_tensor(input)
        pos = torch.log(torch.clamp(x, min=1e-7) + 1)
        neg = -torch.log(torch.clamp(-x, min=1e-7) + 1)
        return torch.where(x > 0, pos, neg)

    # -- gradients ----------------------------------------------------------------------------
    def compute_critic_grad(self, critic_model, target_critic, state_batch, state_next_rollout_batch, partial_reward_to_go_batch,
                            dVdx_batch, d_batch, weights_batch, global_batch=None):
        """NeuralNetwork.py:150-178 -> (critic_grad, reward_to_go, critic_value, target_critic_value(state)).
        ``global_batch`` is the batch size the loss is averaged over (data-parallel shards pass the global one)."""
        f32 = torch.float32
        s = _as_cuda(state_batch, f32)
        B = s.shape[0]
        sn = _as_cuda(state_next_rollout_batch, f32)
        pr = _as_cuda(partial_reward_to_go_batch, f32).reshape(-1)
        dv = _as_cuda(dVdx_batch, f32)
        d = _as_cuda(d_batch, f32).reshape(-1)
        w = _as_cuda(weights_batch, f32).reshape(-1)
        dev = s.device
        rtg = torch.empty((B, 1), dtype=f32, device=dev)
        V = torch.empty((B, 1), dtype=f32, device=dev)
        Vt = torch.empty((B, 1), dtype=f32, device=dev)
        critic_model.grad.zero_()
        self.last_critic_loss.zero_()
        inv_B = 1.0 / float(global_batch if global_batch is not None else B)
        self.launch_critic_grad(critic_model, target_critic, s, sn, pr, dv, d, w, inv_B, rtg, V, Vt, B)
        return critic_model._grad_views, rtg, V, Vt

    def compute_actor_grad(self, actor_model, critic_model, state_batch, term_batch, batch_size, global_batch=None, return_actions=False):
        """NeuralNetwork.py:180-232 -> actor_grad (list of per-variable views of the gradient block)."""
        s = _as_cuda(state_batch, torch.float32)
        B = s.shape[0]
        if batch_size is None:
            batch_size = self.conf.BATCH_SIZE
        term = _as_cuda(term_batch, torch.float64).reshape(-1)
        assert term.numel() == B
        actions = torch.empty((B, actor_model.na), dtype=torch.float32, device=s.device) if return_actions else None
        actor_model.grad.zero_()
        inv_B = 1.0 / float(global_batch if global_batch is not None else B)
        self.launch_actor_grad(actor_model, critic_model, s, term, inv_B, actions, B)
        if return_actions:
            return actor_model._grad_views, actions
        return actor_model._grad_views
