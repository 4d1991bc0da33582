"""Batched restatements of the reference's observation / action wrappers (SURVEY.md section 8f, N1).

Same class names, constructor arguments, ordering rules and attribute surface as ``mate/wrappers/*.py``;
the difference is where the work happens.  The reference applies every wrapper as NumPy slicing on the joint
observation of ONE environment (``np.hstack``, ``.any(axis=0)``, per-row loops).  Here an observation
wrapper only *registers* its transformation with the environment: all registered transformations are
applied in the reference's order by one CUDA kernel over the ``[B, N, D]`` observation tensors right after
the step kernel (``mate_b200_transform_observations``, ``mate_b200/csrc/mate_wrappers.cuh``), so a stack of
wrappers costs one extra read + write of the observations, not one per wrapper.

    env = mate_b200.make('MultiAgentTracking-v0', config='MATE-4v8-9.yaml', num_envs=65536,
                         wrappers=[mate_b200.SharedFieldOfView, mate_b200.RelativeCoordinates,
                                   mate_b200.RescaledObservation, mate_b200.DiscreteCamera])
"""

import functools

import numpy as np
import torch

from mate_b200 import _abi, constants, spaces

TEAMS = ('both', 'camera', 'target', 'none')


class Wrapper:
    """gym.Wrapper-like forwarding: unknown public attributes resolve on the wrapped environment."""

    def __init__(self, env):
        self.env = env

    def __init_subclass__(cls, **kwargs):
        # remember the constructor arguments of the outermost __init__ call: load_config re-runs it
        super().__init_subclass__(**kwargs)
        init = cls.__dict__.get('__init__')
        if init is None:
            return

        @functools.wraps(init)
        def remembering_init(self, env, *args, **kw):
            if type(self) is cls:
                self.__dict__['_ctor_args'] = (args, kw)
            init(self, env, *args, **kw)

        cls.__init__ = remembering_init

    def __getattr__(self, name):
        if name.startswith('_'):
            raise AttributeError(f"attempted to get missing private attribute '{name}'")
        return getattr(self.env, name)

    @property
    def unwrapped(self):
        return self.env.unwrapped

    def reset(self, **kwargs):
        return self.env.reset(**kwargs)

    def step(self, action):
        return self.env.step(action)

    def joint_observation(self):
        return self.env.joint_observation()

    def load_config(self, config=None):
        """Like every wrapper of the reference (``self.env.load_config(config); self.__init__(self.env, ...)``):
        the wrapped environment is re-initialised first, then this wrapper re-runs its own constructor on it, which
        re-registers observation transformations, rebuilds action tables and spaces and re-binds opponent agents
        to the new simulator."""
        self.env.load_config(config=config)
        args, kw = self.__dict__.get('_ctor_args', ((), {}))
        self.__init__(self.env, *args, **kw)  # pylint: disable=unnecessary-dunder-call

    def close(self):
        return self.env.close()

    def __str__(self):
        return f'<{type(self).__name__}{self.env}>'


def _has_wrapper(env, cls):
    while isinstance(env, Wrapper):
        if isinstance(env, cls):
            return True
        env = env.env
    return False


class _ObservationWrapper(Wrapper):
    """Registers its op codes with the base environment (applied on the GPU after every step)."""

    def _register(self, ops):
        base = self.unwrapped
        base.sim.set_observation_wrappers(list(base.sim._obs_ops) + list(ops))  # pylint: disable=protected-access


class EnhancedObservation(_ObservationWrapper):
    """mate/wrappers/enhanced_observation.py: all observation masks True; targets see the empty status of all
    warehouses."""

    def __init__(self, env, team='both'):
        assert team in TEAMS, f'Invalid argument team {team!r}. Expect one of {TEAMS}.'
        assert not _has_wrapper(env, RelativeCoordinates), f'You should use wrapper `{type(self)}` before `RelativeCoordinates`.'
        assert not _has_wrapper(env, RescaledObservation), f'You should use wrapper `{type(self)}` before `RescaledObservation`.'
        super().__init__(env)
        self.team = team
        self.enhanced_camera = team in ('camera', 'both')
        self.enhanced_target = team in ('target', 'both')
        ops = []
        if self.enhanced_camera and env.num_cameras > 0:
            ops.append(_abi.OBS_ENHANCED_CAMERA)
        if self.enhanced_target:
            ops.append(_abi.OBS_ENHANCED_TARGET)
        self._register(ops)

    def __str__(self):
        return f'<{type(self).__name__}(team={self.team}){self.env}>'


class SharedFieldOfView(_ObservationWrapper):
    """mate/wrappers/shared_field_of_view.py: "or" of the view masks of the agents of a team."""

    def __init__(self, env, team='both'):
        assert team in TEAMS, f'Invalid argument team {team!r}. Expect one of {TEAMS}.'
        assert not _has_wrapper(env, RelativeCoordinates), f'You should use wrapper `{type(self)}` before `RelativeCoordinates`.'
        assert not _has_wrapper(env, RescaledObservation), f'You should use wrapper `{type(self)}` before `RescaledObservation`.'
        super().__init__(env)
        self.team = team
        self.shared_camera = team in ('camera', 'both')
        self.shared_target = team in ('target', 'both')
        ops = []
        if self.shared_camera and env.num_cameras > 0:
            ops.append(_abi.OBS_SHARED_CAMERA)
        if self.shared_target:
            ops.append(_abi.OBS_SHARED_TARGET)
        self._register(ops)

    def __str__(self):
        return f'<{type(self).__name__}(team={self.team}){self.env}>'


class RelativeCoordinates(_ObservationWrapper):
    """mate/wrappers/relative_coordinates.py: locations of the other (visible) entities and of the warehouses
    relative to the observing agent."""

    def __init__(self, env):
        assert not _has_wrapper(env, RelativeCoordinates), f'You should not use wrapper `{type(self)}` more than once.'
        assert not _has_wrapper(env, RescaledObservation), f'You should use wrapper `{type(self)}` before `RescaledObservation`.'
        super().__init__(env)
        self._register([_abi.OBS_RELATIVE])


class RescaledObservation(_ObservationWrapper):
    """mate/wrappers/rescaled_observation.py: all entity states rescaled to [-1, +1]."""

    def __init__(self, env):
        assert not _has_wrapper(env, RescaledObservation), f'You should not use wrapper `{type(self)}` more than once.'
        super().__init__(env)
        base = self.unwrapped
        from mate_b200.sim import rescale_tables  # pylint: disable=import-outside-toplevel

        cam_t, tgt_t = rescale_tables(base.num_cameras, base.num_targets, base.num_obstacles)

        def rescaled(space, table):
            t = table.astype(np.float64)
            low = np.where(np.isfinite(space.low), space.low * t[:, 0] + t[:, 1], space.low)
            high = np.where(np.isfinite(space.high), space.high * t[:, 0] + t[:, 1], space.high)
            return spaces.Box(low=low, high=high)

        self.camera_observation_space = rescaled(base.camera_observation_space, cam_t)
        self.target_observation_space = rescaled(base.target_observation_space, tgt_t)
        self.camera_joint_observation_space = spaces.Tuple((self.camera_observation_space,) * base.num_cameras)
        self.target_joint_observation_space = spaces.Tuple((self.target_observation_space,) * base.num_targets)
        self.observation_space = spaces.Tuple((self.camera_joint_observation_space, self.target_joint_observation_space))
        self._register([_abi.OBS_RESCALED])


def camera_action_grid(levels):
    """mate/wrappers/discrete_action_spaces.py:98-117: action_grid[i + levels * j] = (x_i, y_j) in [-1, 1]^2."""
    ticks = np.linspace(start=-1.0, stop=+1.0, num=levels, endpoint=True)
    return np.stack(np.meshgrid(ticks, ticks), axis=-1).reshape(-1, 2)


def target_action_grid(levels):
    """mate/wrappers/discrete_action_spaces.py:204-228: the square grid mapped into the unit disc."""
    grid = camera_action_grid(levels)
    angle = np.arctan2(grid[..., -1], grid[..., 0])
    bound = 1.0 / np.cos(np.pi * ((angle / np.pi + 0.25) % 0.5 - 0.25))
    return grid / bound[..., np.newaxis]


class _DiscreteActions(Wrapper):
    def _table(self, grid):
        return torch.from_numpy(np.ascontiguousarray(grid, dtype=np.float32)).to(self.unwrapped.device)

    def _decode(self, index, table):
        base = self.unwrapped
        index = torch.as_tensor(np.asarray(index) if not torch.is_tensor(index) else index)
        return base.sim.decode_actions(index.to(base.device), table)


class DiscreteCamera(_DiscreteActions):
    """mate/wrappers/discrete_action_spaces.py:21-117: cameras use a levels x levels grid of discrete actions."""

    def __init__(self, env, levels=5):
        assert not _has_wrapper(env, DiscreteCamera), f'You should not use wrapper `{type(self)}` more than once.'
        assert levels >= 3 and levels % 2 == 1, f'The discrete level must be an odd number that not less than 3. Got levels = {levels}.'
        assert env.num_cameras > 0, 'There must be at least one camera in the environment.'
        super().__init__(env)
        self.levels = levels
        self.camera_action_space = spaces.Discrete(levels * levels)
        self.camera_joint_action_space = spaces.Tuple((self.camera_action_space,) * env.num_cameras)
        self.action_space = spaces.Tuple((self.camera_joint_action_space, env.target_joint_action_space))
        self.action_high = np.asarray([env.camera_rotation_step, env.camera_zooming_step], dtype=np.float64)
        self.normalized_action_grid = camera_action_grid(levels)
        self.action_grid = self.action_high * self.normalized_action_grid
        self._device_table = self._table(self.action_grid)

    def action(self, action):
        camera_joint_action, target_joint_action = action
        return self._decode(camera_joint_action, self._device_table), target_joint_action

    def step(self, action):
        return self.env.step(self.action(action))


class DiscreteTarget(_DiscreteActions):
    """mate/wrappers/discrete_action_spaces.py:127-228: targets use a levels x levels grid of discrete actions."""

    def __init__(self, env, levels=5):
        assert not _has_wrapper(env, DiscreteTarget), f'You should not use wrapper `{type(self)}` more than once.'
        assert levels >= 3 and levels % 2 == 1, f'The discrete level must be an odd number that not less than 3. Got levels = {levels}.'
        super().__init__(env)
        self.levels = levels
        self.target_action_space = spaces.Discrete(levels * levels)
        self.target_joint_action_space = spaces.Tuple((self.target_action_space,) * env.num_targets)
        self.action_space = spaces.Tuple((env.camera_joint_action_space, self.target_joint_action_space))
        self.action_high = np.asarray([env.target_step_size, env.target_step_size], dtype=np.float64)
        self.normalized_action_grid = target_action_grid(levels)
        self.action_grid = self.action_high * self.normalized_action_grid
        self._device_table = self._table(self.action_grid)

    def action(self, action):
        camera_joint_action, target_joint_action = action
        return camera_joint_action, self._decode(target_joint_action, self._device_table)

    def step(self, action):
        return self.env.step(self.action(action))


class RepeatedRewardIndividualDone(Wrapper):
    """mate/wrappers/repeated_reward_individual_done.py: the team rewards repeated per agent and a done flag per
    agent (targets: ``target_dones`` if ``target_done_at_destination``)."""

    def __init__(self, env, target_done_at_destination=False):
        assert not _has_wrapper(env, RepeatedRewardIndividualDone), f'You should not use wrapper `{type(self)}` more than once.'
        super().__init__(env)
        self.target_done_at_destination = target_done_at_destination

    def step(self, action):
        observation, (camera_team_reward, target_team_reward), done, info = self.env.step(action)
        base = self.unwrapped
        nc, nt = base.num_cameras, base.num_targets
        if base.batched:
            done_t = torch.as_tensor(done)
            if self.target_done_at_destination:
                target_dones = base.target_dones.to(done_t.dtype)
            else:
                target_dones = done_t.unsqueeze(-1).expand(-1, nt)
            reward = (camera_team_reward.unsqueeze(-1).expand(-1, nc), target_team_reward.unsqueeze(-1).expand(-1, nt))
            return observation, reward, (done_t.unsqueeze(-1).expand(-1, nc), target_dones), info
        target_dones = [bool(x) for x in np.asarray(base.target_dones).reshape(-1)] if self.target_done_at_destination else [done] * nt
        reward = ([camera_team_reward] * nc, [target_team_reward] * nt)
        return observation, reward, ([done] * nc, target_dones), info


# ------------------------------------------------------------------------------------------------------------
# SURVEY.md section 8f, N3: MoreTrainingInformation and the auxiliary-reward wrappers.  The per-agent terms come
# from ONE kernel per step over the auxiliary outputs of the step kernel (``mate_b200_auxiliary_terms``); the
# wrappers only combine columns of that tensor.  Batched: rewards / infos are ``[B, N]`` CUDA tensors (infos: two
# dicts of tensors); reference-compatible single env: Python floats and the reference's list-of-dict infos.
# ------------------------------------------------------------------------------------------------------------

CAMERA_REWARD_KEYS = ('raw_reward', 'coverage_rate', 'real_coverage_rate', 'mean_transport_rate',
                      'soft_coverage_score', 'num_tracked', 'baseline')
TARGET_REWARD_KEYS = ('raw_reward', 'coverage_rate', 'real_coverage_rate', 'mean_transport_rate',
                      'normalized_goal_distance', 'sparse_delivery', 'soft_coverage_score', 'is_tracked',
                      'is_colliding', 'baseline')
_REDUCERS = {
    'mean': lambda x: x.mean(dim=-1, keepdim=True), 'sum': lambda x: x.sum(dim=-1, keepdim=True),
    'max': lambda x: x.max(dim=-1, keepdim=True).values, 'min': lambda x: x.min(dim=-1, keepdim=True).values,
}


def _update_infos(base, infos, per_agent, shared=None):
    """Merge ``{key: [B, N] tensor}`` into the infos of one team (dict of tensors, or the reference's list of dicts)."""
    if base.batched:
        infos.update(per_agent)
        if shared:
            infos.update(shared)
        return
    host = {k: v[0].tolist() for k, v in per_agent.items()}
    for i, info in enumerate(infos):
        for k, values in host.items():
            info[k] = values[i]
        if shared:
            info.update(shared)


class MoreTrainingInformation(Wrapper):
    """mate/wrappers/more_training_information.py: more entries in the info dicts.  Cameras: ``num_tracked``,
    ``is_sensed``; targets: ``goal``, ``goal_distance``, ``warehouse_distances``, ``individual_done``, ``is_tracked``,
    ``is_colliding``; both: the private states of all agents and the view masks.  The entries that need the cargo
    tables / the global state on the host (``state``, ``remaining_cargoes``, ``remaining_cargo_counts``,
    ``awaiting_cargo_counts``, ``obstacle_states``) cost a device synchronisation and are added only with
    ``full_observability=True`` (the default for the reference-compatible single env)."""

    def __init__(self, env, full_observability=None):
        assert not _has_wrapper(env, MoreTrainingInformation), f'You should not use wrapper `{type(self)}` more than once.'
        super().__init__(env)
        base = self.unwrapped
        self.full_observability = (not base.batched) if full_observability is None else bool(full_observability)

    def step(self, action):
        results = self.env.step(action)
        (camera_joint_observation, target_joint_observation), _, _, (camera_infos, target_infos) = results
        base = self.unwrapped
        cam_terms, tgt_terms = base.auxiliary_terms()
        aux = base._aux  # pylint: disable=protected-access
        if base.num_cameras:
            _update_infos(base, camera_infos, {'num_tracked': cam_terms[..., 5].long(), 'is_sensed': cam_terms[..., 7] != 0})
        _update_infos(base, target_infos, {
            'goal': tgt_terms[..., 10].long(), 'goal_distance': tgt_terms[..., 11], 'warehouse_distances': tgt_terms[..., 12:16],
            'individual_done': tgt_terms[..., 5] != 0, 'is_tracked': tgt_terms[..., 7] != 0, 'is_colliding': tgt_terms[..., 8] != 0,
        })
        # full observability (more_training_information.py:84-98)
        cam_self = slice(constants.PRESERVED_DIM, constants.PRESERVED_DIM + constants.CAMERA_STATE_DIM_PRIVATE)
        tgt_self = slice(constants.PRESERVED_DIM, constants.PRESERVED_DIM + constants.TARGET_STATE_DIM_PRIVATE)
        shared = {
            'camera_target_view_mask': aux['mask_ct'].bool(), 'camera_obstacle_view_mask': aux['mask_co'].bool(),
            'target_camera_view_mask': aux['mask_tc'].bool(), 'target_obstacle_view_mask': aux['mask_to'].bool(),
            'target_target_view_mask': aux['mask_tt'].bool(),
        }
        if base.batched:   # a team that is not observed (observed_team) has no rows to take its states from
            if camera_joint_observation is not None:
                shared['camera_states'] = camera_joint_observation[..., cam_self]
            if target_joint_observation is not None:
                shared['target_states'] = target_joint_observation[..., tgt_self]
        else:
            shared = {k: v[0].cpu().numpy() for k, v in shared.items()}
            shared['camera_states'] = np.array(camera_joint_observation[..., cam_self])
            shared['target_states'] = np.array(target_joint_observation[..., tgt_self])
        if self.full_observability:
            remaining = np.asarray(base.remaining_cargoes)
            shared.update(state=base.state(), obstacle_states=np.asarray(base.obstacle_states), remaining_cargoes=remaining,
                          remaining_cargo_counts=remaining.sum(axis=-1), awaiting_cargo_counts=np.asarray(base.awaiting_cargo_counts))
        if base.batched:
            camera_infos.update(shared)
            target_infos.update(shared)
        else:
            for info in list(camera_infos) + list(target_infos):
                info.update({k: (v.copy() if hasattr(v, 'copy') else v) for k, v in shared.items()})
        return results


class _AuxiliaryRewards(Wrapper):
    """Weighted sum of per-agent reward terms (shared implementation of the two wrappers below)."""

    ACCEPTABLE_KEYS = ()
    TEAM = 0   # index into the (camera, target) tuples

    def __init__(self, env, coefficients, reduction='none'):
        cls = type(self)
        assert _has_wrapper(env, RepeatedRewardIndividualDone), (
            f'You should use wrapper `{cls}` with wrapper `RepeatedRewardIndividualDone`. '
            f'Please wrap the environment with wrapper `RepeatedRewardIndividualDone` first. Got env = {env}.')
        assert not _has_wrapper(env, cls), f'You should not use wrapper `{cls}` more than once. Got env = {env}.'
        assert reduction in ('mean', 'sum', 'max', 'min', 'none'), f'Invalid reduction method {reduction}.'
        assert set(self.ACCEPTABLE_KEYS).issuperset(coefficients.keys()), (
            f'The coefficient mapping only accepts keys in {self.ACCEPTABLE_KEYS}. '
            f'Got list(coefficients.keys()) = {list(coefficients.keys())}.')
        self.coefficients = {}
        for key, coefficient in coefficients.items():
            assert callable(coefficient) or isinstance(coefficient, (float, int)), (
                f'The argument `coefficient` should be a callable function or a float number. '
                f'Got coefficients[{key!r}] = {coefficient!r}.')
            self.coefficients[key] = coefficient if not isinstance(coefficient, int) else float(coefficient)
        super().__init__(env)
        self.episode_id = -1
        self.reduction = reduction
        if 'soft_coverage_score' in self.coefficients:
            assert self.unwrapped.num_cameras > 0, "'soft_coverage_score' needs at least one camera."
            self.unwrapped.want_soft_coverage = True   # one more kernel per step (mate_b200_soft_coverage)

    def reset(self, **kwargs):
        self.episode_id += 1
        return self.env.reset(**kwargs)

    def _terms(self, base):
        raise NotImplementedError

    def step(self, action):
        observations, rewards, dones, infos = self.env.step(action)
        base = self.unwrapped
        terms = self._terms(base)                              # [B, N, K] in ACCEPTABLE_KEYS order
        num_agents = terms.shape[1]
        team_infos = infos[self.TEAM]
        if num_agents == 0:
            return observations, rewards, dones, infos
        raw_reward = terms[..., 0]
        reward = torch.zeros_like(raw_reward)
        per_agent = {}
        episode_step = base._aux['episode_step']  # pylint: disable=protected-access
        for key, coefficient in self.coefficients.items():
            value = terms[..., self.ACCEPTABLE_KEYS.index(key)]
            if callable(coefficient):
                if base.batched:   # vectorised call: agent ids [1, N], episode steps [B, 1], values [B, N]
                    agent_ids = torch.arange(num_agents, device=value.device).unsqueeze(0)
                    coefficient = coefficient(agent_ids, self.episode_id, episode_step.unsqueeze(-1), raw_reward, value)
                else:              # the reference's call, one agent at a time
                    coefficient = torch.tensor([[coefficient(i, self.episode_id, int(episode_step[0]), float(raw_reward[0, i]), float(value[0, i]))
                                                 for i in range(num_agents)]], dtype=value.dtype, device=value.device)
            reward = reward + coefficient * value
            per_agent.setdefault(key, value)
            per_agent[f'auxiliary_reward_{key}'] = value
            per_agent[f'reward_coefficient_{key}'] = coefficient if torch.is_tensor(coefficient) else torch.full_like(value, float(coefficient))
        per_agent['reward'] = reward
        if self.reduction in _REDUCERS:
            reward = _REDUCERS[self.reduction](reward).expand(-1, num_agents)
            per_agent['shared_reward'] = reward
        if base.batched:
            for key in self.coefficients:   # info.setdefault(key, ...): keep what an inner wrapper / the env already put there
                if key in team_infos:
                    per_agent.pop(key, None)
            team_infos.update(per_agent)
            team_reward = reward
        else:
            host = {k: v[0].tolist() for k, v in per_agent.items()}
            for i, info in enumerate(team_infos):
                for k, values in host.items():
                    if k in self.coefficients:
                        info.setdefault(k, values[i])
                    else:
                        info[k] = values[i]
            team_reward = reward[0].tolist()
        rewards = (team_reward, rewards[1]) if self.TEAM == 0 else (rewards[0], team_reward)
        return observations, rewards, dones, infos


class AuxiliaryCameraRewards(_AuxiliaryRewards):
    """mate/wrappers/auxiliary_camera_rewards.py: weighted sum of ``raw_reward``, ``coverage_rate``,
    ``real_coverage_rate``, ``mean_transport_rate``, ``soft_coverage_score``, ``num_tracked`` and ``baseline`` per
    camera."""

    ACCEPTABLE_KEYS = CAMERA_REWARD_KEYS
    TEAM = 0

    def _terms(self, base):
        return base.auxiliary_terms()[0][..., :len(CAMERA_REWARD_KEYS)]


class AuxiliaryTargetRewards(_AuxiliaryRewards):
    """mate/wrappers/auxiliary_target_rewards.py: weighted sum of ``raw_reward``, ``coverage_rate``,
    ``real_coverage_rate``, ``mean_transport_rate``, ``normalized_goal_distance``, ``sparse_delivery``,
    ``soft_coverage_score``, ``is_tracked``, ``is_colliding`` and ``baseline`` per target."""

    ACCEPTABLE_KEYS = TARGET_REWARD_KEYS
    TEAM = 1

    def _terms(self, base):
        return base.auxiliary_terms()[1][..., :len(TARGET_REWARD_KEYS)]


# ------------------------------------------------------------------------------------------------------------
# Communication wrappers (mate/wrappers/message_filter.py and its subclasses; DESIGN.md section 7h).  Batched, the
# only messages are those the greedy teams behind MultiCamera / MultiTarget exchange inside their kernels: each wrapper
# merges its rule into the environment's ``message_rules`` and registers them with the simulator, in both modes.  In
# the single-environment mode the wrappers also filter the host ``Message`` traffic in ``send_messages``.
# ------------------------------------------------------------------------------------------------------------

class _CommunicationWrapper(Wrapper):
    """A message filter of the reference: a routed message (broadcasts are one copy per teammate, the sender's own
    included) reaches its recipient iff every communication wrapper of the stack lets it through."""

    def __init__(self, env):
        assert not _has_wrapper(env, MultiCamera) and not _has_wrapper(env, MultiTarget), (
            f'You should use wrapper `{type(self)}` before `MultiCamera` / `MultiTarget`: the single-team wrapper sends '
            f'its opponents\' messages through the environment below it. Please wrap the environment with wrapper '
            f'`{type(self)}` first. Got env = {env}.')
        super().__init__(env)

    def _merge(self, rules):
        raise NotImplementedError

    def _register(self):
        base = self.unwrapped
        self._merge(base.message_rules)
        base.register_message_filter()

    def _delivers(self, base, message):
        raise NotImplementedError

    def send_messages(self, messages):
        base = self.unwrapped
        base._messages_supported()   # pylint: disable=protected-access
        if hasattr(messages, 'sender') and hasattr(messages, 'content'):
            messages = (messages,)
        self.env.send_messages([m for m in base.route_messages(list(messages)) if self._delivers(base, m)])


def _team_of(message):
    from mate_b200 import constants as consts   # pylint: disable=import-outside-toplevel

    return consts._team_index(message.team)   # pylint: disable=protected-access


class RestrictedCommunicationRange(_CommunicationWrapper):
    """mate/wrappers/message_filter.py: a message is delivered iff sender and recipient are at most ``range_limit``
    apart (both teams)."""

    def __init__(self, env, range_limit):
        assert range_limit >= 0, f'The argument `range_limit` should be non-negative. Got range_limit = {range_limit}.'
        super().__init__(env)
        self.range_limit = float(range_limit)
        self._register()

    def _merge(self, rules):
        rules['range_limit'] = [min(limit, self.range_limit) for limit in rules['range_limit']]

    @staticmethod
    def within(a, b, range_limit):
        """The kernels' test: fp64 distance without fused multiply-add, ``<=`` the limit."""
        dx, dy = float(a[0]) - float(b[0]), float(a[1]) - float(b[1])
        return float(np.sqrt(dx * dx + dy * dy)) <= range_limit

    def _delivers(self, base, message):
        agents = base.cameras if _team_of(message) == 0 else base.targets
        return self.within(agents[message.sender].location, agents[message.recipient].location, self.range_limit)


class RandomMessageDropout(_CommunicationWrapper):
    """mate/wrappers/message_filter.py: every message is dropped independently with probability ``dropout_rate``.
    Batched, the draws are Philox streams of the simulator (keyed on its seed and the global environment index);
    in the single-environment mode they come from this wrapper's own ``np_random``."""

    def __init__(self, env, dropout_rate):
        assert 0.0 <= dropout_rate <= 1.0, f'The argument `dropout_rate` should be in [0, 1]. Got dropout_rate = {dropout_rate}.'
        super().__init__(env)
        self.dropout_rate = float(dropout_rate)
        self.np_random = np.random.RandomState(0)
        self._register()

    def seed(self, seed=None):
        self.np_random = np.random.RandomState(seed)
        return self.env.seed(seed)

    def _merge(self, rules):
        rules['keep_probability'] = [keep * (1.0 - self.dropout_rate) for keep in rules['keep_probability']]

    def _delivers(self, base, message):
        return self.np_random.random_sample() >= self.dropout_rate


class NoCommunication(_CommunicationWrapper):
    """mate/wrappers/message_filter.py: drop every message of the named team(s)."""

    def __init__(self, env, team='both'):
        assert team in TEAMS, f'Invalid argument team {team!r}. Expect one of {TEAMS}.'
        super().__init__(env)
        self.team = team
        self.no_camera_communication = team in ('camera', 'both')
        self.no_target_communication = team in ('target', 'both')
        self._register()

    def _merge(self, rules):
        for t, off in enumerate((self.no_camera_communication, self.no_target_communication)):
            if off:
                rules['keep_probability'][t] = 0.0

    def _delivers(self, base, message):
        return not (self.no_camera_communication, self.no_target_communication)[_team_of(message)]

    def __str__(self):
        return f'<{type(self).__name__}(team={self.team}){self.env}>'


# ------------------------------------------------------------------------------------------------------------
# SURVEY.md section 8f, N4: single-team wrapper with a batched built-in opponent.
# ------------------------------------------------------------------------------------------------------------

class _SingleTeamSnapshot:
    """``save_state`` / ``load_state`` of the single-team wrappers: besides the environment they carry the per-environment
    state of the opponent agent (its memory, gathered / scattered along the memory's environment axis with the
    snapshot's index map) and the pending reset mask; the agent's step serial is restored on resume only.  Both teams'
    communication totals travel with the environment's part of the snapshot."""

    _MEMORY_AXIS = None   # environment axis of the agent's field-major memory tensor
    _TEAM = None          # index of this wrapper's team in the joint (camera, target) tuples

    def _pending_resets(self):
        base = self.unwrapped
        if self._reset_mask is True:
            return torch.ones(base.num_envs, dtype=torch.uint8, device=base.device)
        if self._reset_mask is None:
            return torch.zeros(base.num_envs, dtype=torch.uint8, device=base.device)
        return torch.as_tensor(self._reset_mask, device=base.device).to(torch.uint8).clone()

    def save_state(self, envs=None):
        base = self.unwrapped
        snapshot = self.env.save_state(envs)
        agent = self.opponent_agent
        memory, pending = agent._memory, self._pending_resets()   # pylint: disable=protected-access
        if envs is not None:   # out-of-range device indices: the kernel leaves those entries unwritten, here they are clamped
            index = base.sim._index_map(envs, 'envs', None, 0, base.num_envs).long().clamp_(0, base.num_envs - 1)  # pylint: disable=protected-access
            memory, pending = memory.index_select(self._MEMORY_AXIS, index), pending.index_select(0, index)
        snapshot.extras['opponent'] = {'memory': memory.clone(), 'reset_mask': pending.clone(), 'serial': agent._serial}  # pylint: disable=protected-access
        return snapshot

    def load_state(self, snapshot, src=None, resume=False):
        base = self.unwrapped
        joint_observation = self.env.load_state(snapshot, src=src, resume=resume)
        saved = snapshot.extras['opponent']
        agent = self.opponent_agent
        memory, pending = agent._memory, self._pending_resets()   # pylint: disable=protected-access
        saved_memory, saved_pending = saved['memory'].to(memory.device), saved['reset_mask'].to(pending.device)
        if src is None:
            memory.copy_(saved_memory)
            pending = saved_pending.clone()
        else:
            index = base.sim._index_map(src, 'src', base.num_envs, -(1 << 31), snapshot.count).long()  # pylint: disable=protected-access
            keep = (index < 0) | (index >= snapshot.count)
            index = index.clamp(0, snapshot.count - 1)
            shape = [1] * memory.dim()
            shape[self._MEMORY_AXIS] = -1
            memory.copy_(torch.where(keep.view(shape), memory, saved_memory.index_select(self._MEMORY_AXIS, index)))
            pending = torch.where(keep, pending, saved_pending.index_select(0, index))
        self._reset_mask = pending
        if resume:
            agent._serial = saved['serial']   # pylint: disable=protected-access
        self.opponent_infos = None
        self.opponent_joint_observation = joint_observation[1 - self._TEAM]
        return joint_observation[self._TEAM]


class MultiCamera(_SingleTeamSnapshot, Wrapper):
    """mate/wrappers/single_team.py:281-292: a single-team multi-agent environment for the camera team; the targets
    are played by ``target_agent`` (``mate_b200.agents.GreedyTargetAgent``), whose whole team acts in one kernel per
    step on the GPU.  ``reset`` returns the camera joint observation, ``step(camera_joint_action)`` returns
    ``(camera_joint_observation, camera_reward, done, camera_infos)``."""

    _MEMORY_AXIS = 2   # GreedyTargetAgent memory [6, Nt, B]
    _TEAM = 0

    def __init__(self, env, target_agent):
        from mate_b200 import agents  # pylint: disable=import-outside-toplevel

        assert isinstance(target_agent, agents.TargetAgentBase), (
            f'You should provide an instance of target agent. Got target_agent = {target_agent!r}.')
        assert not _has_wrapper(env, MultiCamera), f'You should not use wrapper `{type(self)}` more than once.'
        assert env.num_cameras > 0, 'There must be at least one camera in the environment.'
        if env.unwrapped.observed_team not in ('both', 'camera'):
            raise ValueError(f'MultiCamera returns the camera rows, but this environment observes '
                             f'{env.unwrapped.observed_team!r} only (use observed_team=\'camera\' or \'both\')')
        super().__init__(env)
        self.opponent_agent = target_agent
        self.num_teammates, self.num_opponents = env.num_cameras, env.num_targets
        self.action_space = env.action_space.spaces[0]
        self.observation_space = env.observation_space.spaces[0]
        self.repeated_reward_individual_done = _has_wrapper(env, RepeatedRewardIndividualDone)
        self.opponent_joint_observation = None
        self.opponent_infos = None
        self._reset_mask = True
        target_agent.bind(self.unwrapped.sim)

    def reset(self, **kwargs):
        joint_observation, self.opponent_joint_observation = self.env.reset(**kwargs)
        self.opponent_infos = None
        self._reset_mask = True          # group_reset(opponent_agents, ...), single_team.py:209-219
        return joint_observation

    def step(self, action):
        base = self.unwrapped
        opponent_joint_action = self.opponent_agent.act(reset_mask=self._reset_mask)
        if not base.batched:
            opponent_joint_action = opponent_joint_action[0].double().cpu().numpy()
        (joint_observation, self.opponent_joint_observation), (reward, _), done, (infos, self.opponent_infos) = \
            self.env.step((action, opponent_joint_action))
        # finished episodes were auto-reset inside the step: their opponents start over on the new state
        self._reset_mask = base.sim.done if base.batched else None
        if self.repeated_reward_individual_done:
            done = done[0]
        return joint_observation, reward, done, infos

    def __str__(self):
        return f'<{type(self).__name__}(opponent={type(self.opponent_agent).__module__}.{type(self.opponent_agent).__name__}){self.env}>'


class MultiTarget(_SingleTeamSnapshot, Wrapper):
    """mate/wrappers/single_team.py:295-306: a single-team multi-agent environment for the target team; the cameras
    are played by ``camera_agent`` (``mate_b200.agents.GreedyCameraAgent``), whose whole team acts in one kernel per
    step on the GPU.  ``reset`` returns the target joint observation, ``step(target_joint_action)`` returns
    ``(target_joint_observation, target_reward, done, target_infos)``."""

    _MEMORY_AXIS = 1   # GreedyCameraAgent memory [M, B, Nc]
    _TEAM = 1

    def __init__(self, env, camera_agent):
        from mate_b200 import agents  # pylint: disable=import-outside-toplevel

        assert isinstance(camera_agent, agents.CameraAgentBase), (
            f'You should provide an instance of camera agent. Got camera_agent = {camera_agent!r}.')
        assert not _has_wrapper(env, MultiTarget) and not _has_wrapper(env, MultiCamera), (
            f'You should not use wrapper `{type(self)}` with another single-team wrapper.')
        assert env.num_cameras > 0, 'There must be at least one camera in the environment.'
        if env.unwrapped.observed_team != 'both':
            # the learning targets need their own rows, and the greedy camera team reads its target flags from the camera
            # rows (_tracked_flags): skipping those would need the flags as a separate output of the step kernel
            raise ValueError(f'MultiTarget needs the target rows it returns and the camera rows: the greedy camera team '
                             f'reads its target flags from them (_tracked_flags); this environment observes '
                             f'{env.unwrapped.observed_team!r} only (use observed_team=\'both\')')
        super().__init__(env)
        self.opponent_agent = camera_agent
        self.num_teammates, self.num_opponents = env.num_targets, env.num_cameras
        self.action_space = env.action_space.spaces[1]
        self.observation_space = env.observation_space.spaces[1]
        self.repeated_reward_individual_done = _has_wrapper(env, RepeatedRewardIndividualDone)
        self.opponent_joint_observation = None
        self.opponent_infos = None
        self._reset_mask = True
        camera_agent.bind(self.unwrapped.sim)

    def reset(self, **kwargs):
        self.opponent_joint_observation, joint_observation = self.env.reset(**kwargs)
        self.opponent_infos = None
        self._reset_mask = True
        return joint_observation

    def _tracked_flags(self):
        """Target flags of the cameras' current observations ``[B, Nc, Nt]`` (also right for environments that were
        auto-reset in the last step, whose auxiliary masks still describe the finished step)."""
        base = self.unwrapped
        mask = constants.camera_observation_slices_of(base.num_cameras, base.num_targets, base.num_obstacles)['opponent_mask']
        flags = base.sim.cam_obs[..., mask]
        return (flags > 0.5).to(torch.uint8)

    def step(self, action):
        base = self.unwrapped
        opponent_joint_action = self.opponent_agent.act(self._tracked_flags(), reset_mask=self._reset_mask)
        if not base.batched:
            opponent_joint_action = opponent_joint_action[0].double().cpu().numpy()
        (self.opponent_joint_observation, joint_observation), (_, reward), done, (self.opponent_infos, infos) = \
            self.env.step((opponent_joint_action, action))
        self._reset_mask = base.sim.done if base.batched else None
        if self.repeated_reward_individual_done:
            done = done[1]
        return joint_observation, reward, done, infos

    def __str__(self):
        return f'<{type(self).__name__}(opponent={type(self.opponent_agent).__module__}.{type(self.opponent_agent).__name__}){self.env}>'
