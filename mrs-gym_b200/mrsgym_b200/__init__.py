"""mrsgym_b200 -- B200-native implementation of the mrs-gym per-step hot path.

    import mrsgym_b200 as mrsgym
    env = mrsgym.make('mrs-v0', N_AGENTS=8, N_ENVS=65536, K_HOPS=3, COMM_RANGE=2.0, ACTION_TYPE='set_speeds')
    X, reward, done, info = env.step(actions)        # info['A'] is the adjacency history

`make` works without gym; when gym / gymnasium is importable the id 'mrs-v0' is also
registered there (reference: /root/reference/mrsgym/__init__.py:13-16).
"""
from . import _abi
from ._abi import MrsError
from .core import Swarm, Neighbors, shard_range
from .env import MRS, Environment, AgentBatch
from .spawn import DefaultSpawn, sample_start_pos
from .rollout import rollout, reynolds_policy, to_trainer_history, save_dataset, ClosedLoopGraph
from .wrappers import MRS_RLlib, MRS_RLlib_MultiAgent

_REGISTRY = {'mrs-v0': MRS, 'mrs-rllib-v0': MRS_RLlib, 'mrs-rllib-multiagent-v0': MRS_RLlib_MultiAgent}


def make(env_id, **kwargs):
    """gym.make stand-in: make('mrs-v0', **kwargs) -> MRS(**kwargs)."""
    if env_id not in _REGISTRY:
        raise KeyError('unknown environment id %r (known: %s)' % (env_id, ', '.join(_REGISTRY)))
    if env_id != 'mrs-v0':
        return _REGISTRY[env_id](kwargs.get('config', kwargs))
    return _REGISTRY[env_id](**kwargs)


def _register():
    for modname in ('gymnasium', 'gym'):
        try:
            mod = __import__(modname + '.envs.registration', fromlist=['register'])
            mod.register(id='mrs-v0', entry_point='mrsgym_b200:MRS')
            mod.register(id='mrs-rllib-v0', entry_point='mrsgym_b200:MRS_RLlib')
            mod.register(id='mrs-rllib-multiagent-v0', entry_point='mrsgym_b200:MRS_RLlib_MultiAgent')
        except Exception:
            pass


_register()
