"""Which kernel ``RL_AC._launch_rollout`` runs for an episode, an engine, the actor's kind and the system's inputs
(``RL_AC._rollout_kernel``).  No GPU needed: a stub RL_AC with only an actor description."""
from types import SimpleNamespace

import pytest

ENGINES = ('tc', 'tf32', 'fma')


def stub(ns, kind='actor'):
    from cacto_b200.RL import RL_AC
    rl = RL_AC.__new__(RL_AC)
    rl.actor_model = SimpleNamespace(kind=kind, ns=ns)
    return rl


CASES = ([(0, kind, ns, e, 'fma') for kind in ('actor', 'actor_width') for ns in (7, 13) for e in ENGINES + (None,)] +
         [(1, 'actor_width', ns, e, 'width') for ns in (7, 13) for e in ENGINES + (None,)] +
         [(1, 'actor', 7, 'tc', 'tc'), (1, 'actor', 13, 'tc', 'tf32'), (1, 'actor', 7, None, 'tc'), (1, 'actor', 13, None, 'tf32')] +
         [(1, 'actor', ns, e, e) for ns in (7, 13) for e in ('tf32', 'fma')])


@pytest.mark.parametrize('ep,kind,ns,engine,kernel', CASES)
def test_rollout_kernel(ep, kind, ns, engine, kernel):
    assert stub(ns, kind)._rollout_kernel(ep, engine) == kernel


@pytest.mark.parametrize('engine', ['tc2', 'bogus'])
@pytest.mark.parametrize('ep', [0, 1])
def test_unknown_rollout_engine_is_refused(ep, engine):
    with pytest.raises(ValueError):
        stub(7)._rollout_kernel(ep, engine)
