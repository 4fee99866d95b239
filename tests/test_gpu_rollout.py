"""Fused actor + dynamics rollout kernel (K1) against the oracle's restatement of RL_AC.create_TO_init and the
reference-generated goldens."""
import numpy as np
import pytest
import torch

from cacto_b200.conf import SYSTEM_IDS, get_conf
from conftest import golden
from oracle import nn as onn
from oracle import rtg as ortg
from oracle import systems as osys

pytestmark = pytest.mark.gpu


def setup(system, seed=0):
    from cacto_b200 import environment as genv
    from cacto_b200.NeuralNetwork import NN
    from cacto_b200.RL import RL_AC
    conf = get_conf(system)
    env = genv.make_env(conf)
    rl = RL_AC(env, NN(env, conf, 1e-2, seed=seed), conf, 0)
    rl.setup_model()
    return conf, env, rl


def ics(conf, B, seed):
    rng = np.random.default_rng(seed)
    x = rng.uniform(np.asarray(conf.x_init_min, float), np.asarray(conf.x_init_max, float), (B, conf.nb_state))
    x[:, -1] = conf.dt * np.round(x[:, -1] / conf.dt)
    return x


@pytest.mark.parametrize('system', SYSTEM_IDS)
@pytest.mark.parametrize('ep,engine', [(0, 'fma'), (1, 'fma'), (1, 'tc'), (1, 'tf32')])
def test_rollout_batch_matches_oracle(system, ep, engine):
    """engine 'fma' = fp32 CUDA-core kernel, 'tc' = tcgen05 fp16-split persistent kernel (default), 'tf32' = tcgen05 3xTF32
    kernel (256 rollouts per CTA)."""
    conf, env, rl = setup(system)
    rl.rollout_engine = engine
    B = (70 if engine == 'fma' else 300) if system != 'ur5' else 5      # more than one CTA, ragged tile, mixed horizons
    X0 = ics(conf, B, 3)
    X0[0, -1] = 0.0                            # full horizon
    X0[1, -1] = (conf.NSTEPS - 1) * conf.dt    # one step
    out = rl.rollout_batch(X0, ep)
    states = out['states'].permute(2, 0, 1).cpu().numpy()
    controls = out['controls'].permute(2, 0, 1).cpu().numpy()
    hz = out['horizon'].cpu().numpy()
    assert out['success'].cpu().numpy().all()
    oenv = osys.make_env(conf)
    ap = onn.to_torch(rl.actor_model.get_weights())

    def actor_eval(x):
        with torch.no_grad():
            return onn.actor_forward(ap, torch.tensor(x, dtype=torch.float32), conf).numpy()[0]
    n_check = (B if system != 'ur5' else 3) if engine == 'fma' else min(B, 12)
    check = list(range(n_check)) if engine == 'fma' else [i for i in ([0, 1, 127, 128, 255, 256, B - 1] + list(range(2, 7))) if i < B][:n_check]
    for b in check:
        _, st, ct, T, ok = ortg.create_to_init(conf, oenv, actor_eval, ep, X0[b])
        assert ok == 1 and T == hz[b] == ortg.horizon(conf, X0[b, -1])
        sc = np.abs(st).max(axis=0) + 1e-12
        assert (np.abs(states[b, :T + 1] - st) / sc).max() < 1e-4, (b, T)
        if T > 0:
            assert np.abs(controls[b, :T] - ct).max() <= 1e-4 * max(np.abs(ct).max(), 1e-3)
        assert np.isnan(states[b, T + 1:]).all()          # entries past the horizon are untouched


@pytest.mark.parametrize('system', ['single_integrator', 'car', 'car_park'])
def test_create_TO_init_matches_reference_goldens(system):
    """The reference's own create_TO_init loop (tests/golden/toinit_cases.npz)."""
    g = golden('toinit_cases.npz')
    conf, env, rl = setup(system)
    rl.actor_model.set_weights([g[f'{system}_actor_{i}'] for i in range(6)])
    for k in range(3):
        for ep in (0, 1):
            x0 = g[f'{system}_{k}_{ep}_ics']
            _, st, ct, T, ok = rl.create_TO_init(ep, x0)
            assert ok == 1 and T == int(g[f'{system}_{k}_{ep}_T'])
            ref_s, ref_c = g[f'{system}_{k}_{ep}_states'], g[f'{system}_{k}_{ep}_controls']
            tol = 1e-12 if ep == 0 else 1e-4
            sc = np.abs(ref_s).max(axis=0) + 1e-12
            assert (np.abs(st - ref_s) / sc).max() <= tol
            assert np.abs(ct - ref_c).max() <= tol * max(1.0, np.abs(ref_c).max())


@pytest.mark.parametrize('engine,B', [('tc', 1000), ('tf32', 1000), ('tc', 40000)])
def test_tensor_core_engine_agrees_with_fma_engine(engine, B):
    """Full-size tile coverage: manipulator rollouts with mixed horizons, tensor-core engine vs fp32 FMA engine, same actor.
    B = 40000 gives the persistent 'tc' kernel 313 tiles over 148 CTAs (2-3 tiles per CTA, ragged last tile)."""
    conf, env, rl = setup('manipulator')
    X0 = ics(conf, B, 7)
    a = rl.rollout_batch(X0, 1, engine='fma')
    b = rl.rollout_batch(X0, 1, engine=engine)
    assert bool((torch.isnan(a['states']) == torch.isnan(b['states'])).all())
    m = ~torch.isnan(a['states'])
    assert float((a['states'][m] - b['states'][m]).abs().max()) < 1e-5
    m = ~torch.isnan(a['controls'])
    assert float((a['controls'][m] - b['controls'][m]).abs().max()) < 1e-5
    assert bool((a['success'] == b['success']).all())


@pytest.mark.parametrize('engine', ['fma', 'tc', 'tf32'])
def test_horizon_zero_and_nan_flag(engine):
    conf, env, rl = setup('manipulator')
    rl.rollout_engine = engine
    x0 = ics(conf, 4, 1)
    x0[0, -1] = conf.NSTEPS * conf.dt          # NSTEPS_SH = 0 (RL.py:202-203)
    assert rl.create_TO_init(1, x0[0])[-1] == 0
    x0[1, 0] = np.nan
    out = rl.rollout_batch(x0, 1)
    ok = out['success'].cpu().numpy()
    assert ok[1] == 0 and ok[2] == 1 and ok[3] == 1


def test_rollout_rewards_match_env_step():
    """PLOT.rollout-style rewards (plot_utils.py:261-268): running reward at (x_t, u_t), terminal at x_T."""
    conf, env, rl = setup('manipulator')
    x0 = ics(conf, 6, 2)
    out = rl.rollout_batch(x0, 1, with_reward=True)
    oenv = osys.make_env(conf)
    S = out['states'].permute(2, 0, 1).cpu().numpy()
    U = out['controls'].permute(2, 0, 1).cpu().numpy()
    R = out['rewards'].permute(1, 0).cpu().numpy()
    hz = out['horizon'].cpu().numpy()
    for b in range(6):
        T = hz[b]
        ref = [oenv.reward(conf.cost_weights_running, S[b, t], U[b, t]) for t in range(T)] + [oenv.reward(conf.cost_weights_terminal, S[b, T])]
        np.testing.assert_allclose(R[b, :T + 1], ref, rtol=1e-9, atol=1e-14)


def test_rollout_to_host_modes_agree():
    """Host-to-host rollouts: pipelined sub-batches with strided DMA, zero-copy stores and the staged copy deliver the same
    trajectories (knots inside each horizon; entries past it are unspecified in the staged modes)."""
    conf, env, rl = setup('manipulator')
    B, T, ns, na = 1000, conf.NSTEPS, conf.nb_state, conf.nb_action
    X0 = ics(conf, B, 11)
    ih = torch.as_tensor(X0).pin_memory()
    outs = {}
    for mode in ('pipelined', 'zero_copy', 'staged'):
        st = torch.full((T + 1, ns, B), float('nan'), dtype=torch.float64).pin_memory()
        ct = torch.full((T, na, B), float('nan'), dtype=torch.float64).pin_memory()
        fl = torch.zeros(B, dtype=torch.int32).pin_memory()
        hz = rl.rollout_to_host(ih, 1, st, ct, fl, mode=mode, n_chunks=3)
        outs[mode] = (st.clone(), ct.clone(), fl.clone(), hz)
    ref = rl.rollout_batch(X0, 1)
    hz = ref['horizon'].cpu().numpy()
    knots = np.arange(T + 1)[:, None] <= hz[None, :]
    for mode, (st, ct, fl, h) in outs.items():
        assert (h == hz).all() and bool(fl.all())
        a, b = st.numpy(), ref['states'].cpu().numpy()
        m = np.broadcast_to(knots[:, None, :], a.shape)
        # the sub-batches of the pipelined mode change which tile pipeline runs a rollout: equal to fp32 rounding of the actor
        assert np.abs(a[m] - b[m]).max() < 1e-5
        mc = np.broadcast_to(knots[:-1, None, :] & (np.arange(T)[:, None, None] < hz[None, None, :]), ct.shape)
        assert np.abs(ct.numpy()[mc] - ref['controls'].cpu().numpy()[mc]).max() < 1e-5


def test_rollout_to_host_without_waiting_delivers_the_same_batches():
    """wait=False: two batches in flight on alternating host buffers (the staging slots on the device are shared): each arrives
    complete and bit-identical to the blocking call."""
    conf, env, rl = setup('manipulator')
    B, T, ns, na = 700, conf.NSTEPS, conf.nb_state, conf.nb_action
    ih = [torch.as_tensor(ics(conf, B, 21 + i)).pin_memory() for i in range(3)]
    def bufs():
        return (torch.full((T + 1, ns, B), float('nan'), dtype=torch.float64).pin_memory(),
                torch.full((T, na, B), float('nan'), dtype=torch.float64).pin_memory(), torch.zeros(B, dtype=torch.int32).pin_memory())
    want = []
    for x in ih:
        st, ct, fl = bufs()
        hz = rl.rollout_to_host(x, 1, st, ct, fl, n_chunks=3)
        want.append((st.clone(), ct.clone(), fl.clone(), hz))
    sets = (bufs(), bufs())
    pending, got = None, []
    for k, x in enumerate(ih):
        cur = sets[k & 1]
        h = rl.rollout_to_host(x, 1, cur[0], cur[1], cur[2], n_chunks=3, wait=False)
        if pending is not None:
            hz = pending[0].wait()
            got.append((pending[1][0].clone(), pending[1][1].clone(), pending[1][2].clone(), hz))
        pending = (h, cur)
    hz = pending[0].wait()
    got.append((pending[1][0].clone(), pending[1][1].clone(), pending[1][2].clone(), hz))
    for (st, ct, fl, hz), (st2, ct2, fl2, hz2) in zip(want, got):
        assert (hz == hz2).all() and bool(fl2.all()) and torch.equal(fl, fl2)
        knots = np.arange(T + 1)[:, None] <= hz[None, :]                   # entries past a rollout's horizon are left untouched
        m = np.broadcast_to(knots[:, None, :], st.shape)
        assert np.array_equal(st.numpy()[m], st2.numpy()[m])
        mc = np.broadcast_to((np.arange(T)[:, None] < hz[None, :])[:, None, :], ct.shape)
        assert np.array_equal(ct.numpy()[mc], ct2.numpy()[mc])


def test_rollout_to_host_compact_is_bit_reconstructible():
    """compact=True moves 25 % fewer bytes over PCIe (no time row, controls as the fp32 values the actor produced); the
    reference-shaped arrays ``CompactRollouts`` rebuilds are bit-identical to the full-format transfer of the same batch."""
    from cacto_b200.RL import CompactRollouts
    conf, env, rl = setup('manipulator')
    B, T, ns, na = 900, conf.NSTEPS, conf.nb_state, conf.nb_action
    X0 = ics(conf, B, 31)
    X0[:, -1] = np.random.default_rng(5).integers(0, T, B) * conf.dt          # ragged horizons, non-zero start times
    ih = torch.as_tensor(X0).pin_memory()
    st = torch.full((T + 1, ns, B), float('nan'), dtype=torch.float64).pin_memory()
    ct = torch.full((T, na, B), float('nan'), dtype=torch.float64).pin_memory()
    fl = torch.zeros(B, dtype=torch.int32).pin_memory()
    hz = rl.rollout_to_host(ih, 1, st, ct, fl, n_chunks=3)
    sc = torch.full((T + 1, ns - 1, B), float('nan'), dtype=torch.float64).pin_memory()
    cc = torch.full((T, na, B), float('nan'), dtype=torch.float32).pin_memory()
    fc = torch.zeros(B, dtype=torch.int32).pin_memory()
    hzc = rl.rollout_to_host(ih, 1, sc, cc, fc, n_chunks=3, compact=True)
    assert (hz == hzc).all() and bool(fc.all()) and torch.equal(fl, fc)
    view = CompactRollouts(conf, ih, sc, cc, hzc)
    for b in range(B):
        Tb = int(hz[b])
        assert np.array_equal(view.states(b), st.numpy()[:Tb + 1, :, b])
        assert np.array_equal(view.controls(b), ct.numpy()[:Tb, :, b])
    with pytest.raises(ValueError):
        rl.rollout_to_host(ih, 1, st, ct, fl, compact=True)                    # full-format buffers with compact=True
    with pytest.raises(ValueError):
        rl.rollout_to_host(ih, 1, sc, cc, fc, mode='staged', compact=True)


def test_tc_engine_overflow_falls_back_to_fma():
    """An actor whose hidden activations leave the fp16 range of the 'tc' engine (rollout_tc16.cu: +-2047 after scaling) must not
    change the outcome: the reference aborts on NaN only (RL.py:229-231).  Flagged rollouts are re-run on 'fma'."""
    conf, env, rl = setup('manipulator')
    w = rl.actor_model.get_weights()
    w[0] = w[0] * 3e4                       # first-layer activations ~1e4: beyond the +-2047 the fp16 high part of 32 h1 can hold
    w[2] = w[2] / 3e4                       # keep the actions (and the dynamics) in range
    rl.actor_model.set_weights(w)
    X0 = ics(conf, 300, 11)
    X0[:, -1] = (conf.NSTEPS - 20) * conf.dt
    ref = rl.rollout_batch(X0, 1, engine='fma')
    assert ref['success'].cpu().numpy().all()
    # the raw engine does flag them ...
    dev = ref['states'].device
    T = int(conf.NSTEPS)
    st = torch.full_like(ref['states'], float('nan')); ct = torch.full_like(ref['controls'], float('nan'))
    fl = torch.empty(300, dtype=torch.int32, device=dev)
    rl._launch_rollout(1, torch.as_tensor(X0, device=dev), ref['horizon'], T, st, ct, fl, None, 300, 'tc')
    assert (fl.cpu().numpy() == 0).any(), 'the scaled actor was meant to overflow the fp16 engine'
    # ... and rollout_batch repairs them
    out = rl.rollout_batch(X0, 1, engine='tc')
    assert out['success'].cpu().numpy().all()
    a, b = out['states'].cpu().numpy(), ref['states'].cpu().numpy()
    m = ~np.isnan(b)
    assert (np.isnan(a) == np.isnan(b)).all()
    assert np.abs(a[m] - b[m]).max() <= 1e-4 * np.abs(b[m]).max()
    # host-to-host path
    sh = torch.empty((T + 1, conf.nb_state, 300), dtype=torch.float64).pin_memory()
    ch = torch.empty((T, conf.nb_action, 300), dtype=torch.float64).pin_memory()
    fh = torch.empty(300, dtype=torch.int32).pin_memory()
    rl.rollout_to_host(torch.as_tensor(X0).pin_memory(), 1, sh, ch, fh)
    assert fh.numpy().all()
    hz = ref['horizon'].cpu().numpy()
    for b_ in (0, 150, 299):
        np.testing.assert_allclose(sh[:hz[b_] + 1, :, b_].numpy(), b[:hz[b_] + 1, :, b_], rtol=1e-4, atol=1e-6)

