"""mate_b200: B200-native batched simulator for MATE's ``MultiAgentTracking`` step.

Drop-in for the reference's env entry points (mate/__init__.py:24-101)::

    import mate_b200 as mate
    env = mate.make('MultiAgentTracking-v0', config='MATE-4v8-9.yaml', num_envs=65536)
    cam_obs, tgt_obs = env.reset(seed=0)
    (cam_obs, tgt_obs), (cam_r, tgt_r), done, infos = env.step((cam_act, tgt_act))

The simulation runs in hand-written sm_100a CUDA behind the C ABI of
``include/mate_b200.h``; importing this package does not need a GPU, creating an
environment does (there is no CPU fallback).
"""

from mate_b200 import config, constants
from mate_b200.config import PRESETS, flatten_config, preset, read_config
from mate_b200.constants import *  # noqa: F401,F403
from mate_b200.messages import Message, Team  # noqa: F401

__version__ = '0.1.0'

_REGISTRY = {}


class _Spec:
    def __init__(self, id):  # pylint: disable=redefined-builtin
        self.id = id


def register(id, entry_point, kwargs=None):  # pylint: disable=redefined-builtin
    """Register an environment id (gym.register-like: kwargs are defaults for `make`)."""
    _REGISTRY[id] = (entry_point, dict(kwargs or {}))


def make_environment(config=None, wrappers=(), **kwargs):  # pylint: disable=redefined-outer-name
    """Create a (wrapped) environment (mate/__init__.py:27-43)."""
    from mate_b200.environment import MultiAgentTracking  # pylint: disable=import-outside-toplevel

    env = MultiAgentTracking(config, **kwargs)
    for wrapper in wrappers:
        if not callable(wrapper):
            raise AssertionError(f'You should provide a wrapper class or a callable. Got wrapper = {wrapper!r}.')
        env = wrapper(env)
    return env


def make(id, **kwargs):  # pylint: disable=redefined-builtin
    """``mate.make`` (== ``gym.make`` in the reference): create a registered environment."""
    if id not in _REGISTRY:
        raise KeyError(f'No registered env with id: {id}. Known ids: {sorted(_REGISTRY)}')
    entry_point, defaults = _REGISTRY[id]
    merged = dict(defaults)
    merged.update(kwargs)
    env = entry_point(**merged)
    env.unwrapped.spec = _Spec(id)
    return env


register('MultiAgentTracking-v0', make_environment)
register('MATE-v0', make_environment)
for _nc, _nt in ((4, 2), (4, 4), (4, 8), (8, 8)):
    for _no in (9, 0):
        register(f'MATE-{_nc}v{_nt}-{_no}-v0', make_environment, {'config': f'MATE-{_nc}v{_nt}-{_no}.yaml'})
register('MATE-Navigation-v0', make_environment, {'config': 'MATE-Navigation.yaml'})
del _nc, _nt, _no


_WRAPPERS = ('EnhancedObservation', 'SharedFieldOfView', 'RelativeCoordinates', 'RescaledObservation',
             'DiscreteCamera', 'DiscreteTarget', 'RepeatedRewardIndividualDone', 'MoreTrainingInformation',
             'AuxiliaryCameraRewards', 'AuxiliaryTargetRewards', 'MultiCamera', 'MultiTarget',
             'RestrictedCommunicationRange', 'RandomMessageDropout', 'NoCommunication')
_AGENTS = ('GreedyTargetAgent', 'GreedyCameraAgent', 'TargetAgentBase', 'CameraAgentBase')


def __getattr__(name):
    if name in _WRAPPERS or name == 'wrappers':   # lazy for the same reason as below
        import importlib  # pylint: disable=import-outside-toplevel

        module = importlib.import_module('mate_b200.wrappers')
        return module if name == 'wrappers' else getattr(module, name)
    if name in _AGENTS or name == 'agents':
        import importlib  # pylint: disable=import-outside-toplevel

        module = importlib.import_module('mate_b200.agents')
        return module if name == 'agents' else getattr(module, name)
    if name == 'MultiAgentTracking':   # lazy: importing torch is slow and not needed for config work
        from mate_b200.environment import MultiAgentTracking  # pylint: disable=import-outside-toplevel

        return MultiAgentTracking
    raise AttributeError(name)
