"""``MultiAgentTracking`` over a leading batch-of-environments dimension.

Host-side mirror of the reference's env class (mate/environment.py:288-1560) for the step
path: same constructor arguments (config path / dict / preset name + keyword overrides),
``reset`` / ``step`` / ``seed`` / ``state`` / ``joint_observation`` / ``load_config``, the
joint ``(camera, target)`` tuple layout of observations, actions and rewards, the spaces,
the view-mask / cargo attributes wrappers read, and the reference's error behaviour
(non-finite actions are rejected like ``mate/environment.py:1337-1342``).

Two calling conventions:

* batched (``num_envs=B``): everything is a CUDA tensor with a leading ``B`` dimension;
  ``step`` auto-resets finished episodes (the returned observation is the first one of the
  new episode, rewards/done/infos are those of the finished step); infos are two dicts of
  ``[B]`` tensors instead of ``B * (Nc + Nt)`` Python dicts.
* reference-compatible (``num_envs=None``, the default): one environment, NumPy float64
  arrays, Python floats / bool, list-of-dict infos, and NO auto-reset -- the exact
  types of the reference, so existing single-env user code and wrappers keep working.

All simulation happens in ``libmate_b200.so`` (hand-written sm_100a CUDA); this module only
moves pointers.  There is no CPU fallback.
"""

import copy
from collections import defaultdict, deque
from typing import Any, Dict, Iterable, List, Optional, Tuple, Union

import numpy as np
import torch

from mate_b200 import constants as consts
from mate_b200 import spaces
from mate_b200.config import DEFAULT_CONFIG_FILE, flatten_config, read_config
from mate_b200.entities import CameraView, ObstacleView, TargetView
from mate_b200.messages import Message, Team
from mate_b200.sim import BatchedSim, check_index_map, check_observation_dtype, check_observed_team, check_render_size

__all__ = ['MultiAgentTracking', 'EnvMeta', 'Message', 'Team', 'read_config', 'DEFAULT_CONFIG_FILE']


class EnvMeta(type):
    """``isinstance(wrapped_env, MultiAgentTracking)`` sees through wrappers, like the reference's metaclass
    (mate/environment.py:272-284): any object that reaches a ``MultiAgentTracking`` through a chain of ``.env``
    attributes (``mate_b200.wrappers.Wrapper``, ``gym.Wrapper``) is an instance."""

    def __instancecheck__(cls, instance):
        if super().__instancecheck__(instance):
            return True
        seen = 0
        while hasattr(type(instance), 'env') or 'env' in getattr(instance, '__dict__', {}):
            instance = instance.env
            seen += 1
            if super().__instancecheck__(instance):
                return True
            if seen > 64:
                break
        return False


class MultiAgentTracking(metaclass=EnvMeta):  # pylint: disable=too-many-instance-attributes,too-many-public-methods
    """Batched Multi-Agent Tracking Environment (cameras vs. cargo-hauling targets)."""

    metadata = {'render.modes': ['rgb_array']}
    DEFAULT_CONFIG_FILE = DEFAULT_CONFIG_FILE
    spec = None
    _sim_class = BatchedSim   # the simulator behind the class (tests substitute a recorded one to exercise this host layer without a GPU)

    def __init__(self, config: Optional[Union[Dict[str, Any], str]] = None, num_envs: Optional[int] = None,
                 device: Union[int, str, torch.device] = 0, env_index_base: int = 0,
                 observation_dtype: torch.dtype = torch.float32, observed_team: str = 'both', **kwargs) -> None:
        # observation_dtype: element type of the batched observation tensors, torch.float32 or torch.float16 (the float32
        # rows rounded once to nearest even); the observation spaces keep describing the reference's float64 Boxes
        check_observation_dtype(observation_dtype)
        if num_envs is None and observation_dtype != torch.float32:
            raise ValueError('observation_dtype applies to the batched mode (num_envs=B); the single-environment mode '
                             'returns the float64 NumPy observations of the reference')
        # observed_team: whose observation rows the simulator composes ('both', 'camera' or 'target'); the joint
        # observations carry None in the other team's slot (one team learning against built-in agents)
        check_observed_team(observed_team)
        if num_envs is None and observed_team != 'both':
            raise ValueError("observed_team applies to the batched mode (num_envs=B); the single-environment mode "
                             "observes both teams")
        if config is None:
            config = {} if len(kwargs) > 0 else self.DEFAULT_CONFIG_FILE   # environment.py:338-339
        self._init_args = (config, num_envs, device, env_index_base, dict(kwargs), observation_dtype, observed_team)
        self.config = read_config(config, **kwargs)
        self.flat_config = flatten_config(self.config)
        check_observed_team(observed_team, self.flat_config['num_cameras'])
        self.batched = num_envs is not None
        self.num_envs = int(num_envs) if self.batched else 1
        self.observation_dtype = observation_dtype
        self.observed_team = observed_team
        # the defaults are not passed on: simulator classes substituted for BatchedSim need not know the arguments
        sim_kwargs = {} if observation_dtype == torch.float32 else {'observation_dtype': observation_dtype}
        if observed_team != 'both':
            sim_kwargs['observed_team'] = observed_team
        self.sim = self._sim_class(self.flat_config, self.num_envs, device=device, env_index_base=env_index_base, **sim_kwargs)
        self.device = self.sim.device
        nc, nt, no = self.num_cameras, self.num_targets, self.num_obstacles

        cam = self.flat_config
        self.camera_action_space = spaces.Box(
            low=np.array([-cam['camera_rotation_step'], -cam['camera_zooming_step']]) if nc else np.zeros(2),
            high=np.array([cam['camera_rotation_step'], cam['camera_zooming_step']]) if nc else np.zeros(2))
        step = cam['target_step_size']
        self.target_action_space = spaces.Box(low=np.array([-step, -step]), high=np.array([step, step]))
        self.camera_joint_action_space = spaces.Tuple((self.camera_action_space,) * nc)
        self.target_joint_action_space = spaces.Tuple((self.target_action_space,) * nt)
        self.action_space = spaces.Tuple((self.camera_joint_action_space, self.target_joint_action_space))
        self.camera_observation_space = consts.camera_observation_space_of(nc, nt, no)
        self.target_observation_space = consts.target_observation_space_of(nc, nt, no)
        self.camera_joint_observation_space = spaces.Tuple((self.camera_observation_space,) * nc)
        self.target_joint_observation_space = spaces.Tuple((self.target_observation_space,) * nt)
        self.observation_space = spaces.Tuple((self.camera_joint_observation_space, self.target_joint_observation_space))
        self.state_space = spaces.Box(
            low=np.concatenate([consts.PRESERVED_LOW] + [consts.CAMERA_PRIVATE_LOW] * nc + [consts.TARGET_PRIVATE_LOW] * nt
                               + [consts.OBSTACLE_LOW] * no + [np.zeros(2 * nt + 16)]),
            high=np.concatenate([consts.PRESERVED_HIGH] + [consts.CAMERA_PRIVATE_HIGH] * nc + [consts.TARGET_PRIVATE_HIGH] * nt
                                + [consts.OBSTACLE_HIGH] * no + [np.full(2 * nt + 16, np.inf)]))

        self.freight_scale = float(np.ceil(consts.TERRAIN_WIDTH / self.target_step_size))   # environment.py:521-529
        self.bounty_scale = float(np.ceil(self.freight_scale * self.bounty_factor))
        self.reward_scale = self.freight_scale + self.bounty_scale
        self.max_target_team_episode_reward = self.reward_scale * self.num_cargoes_per_target * nt

        self._seed = 0
        self._np_random = np.random.RandomState(0)
        self._needs_reset = True
        self._step_serial = 0
        self._terms_serial = -1
        self._terms = None
        self.want_soft_coverage = False   # set by an auxiliary-reward wrapper that uses 'soft_coverage_score'
        self._aux = self.sim.alloc_aux()
        self._snapshot_cache = (None, None)
        self._state_serial = 0
        self.cameras = [CameraView(self, c) for c in range(nc)]       # mate/environment.py:392-398
        self.targets = [TargetView(self, t) for t in range(nt)]
        self.obstacles = [ObstacleView(self, o) for o in range(no)]
        self.cameras_ordered, self.targets_ordered, self.obstacles_ordered = self.cameras, self.targets, self.obstacles
        self.preserved_data = np.concatenate([[nc, nt, no, 0.0], consts.WAREHOUSES.ravel(), [consts.WAREHOUSE_RADIUS]]).astype(np.float64)
        self.viewer = None
        self.render_callbacks = {}
        # intra-team messages (mate/environment.py:540-562): host objects of the reference-compatible mode
        self.camera_message_buffer, self.target_message_buffer = defaultdict(list), defaultdict(list)
        self.message_buffers = (self.camera_message_buffer, self.target_message_buffer)
        self.camera_message_queue, self.target_message_queue = defaultdict(deque), defaultdict(deque)
        self.message_queues = (self.camera_message_queue, self.target_message_queue)
        # communication edges: in the single-environment mode the host Message traffic (NumPy, like the reference); in
        # batched mode the traffic of the batched greedy teams, written by their kernels (DESIGN.md section 7h):
        # delivered sets of the team's last call (int64 [B], bit 8 s + r) and per-episode totals (int32 [B, N, N])
        if self.batched:
            self._delivered_bits = tuple(torch.zeros(self.num_envs, dtype=torch.int64, device=self.device) for _ in range(2))
            self._total_edges = tuple(torch.zeros((self.num_envs, n, n), dtype=torch.int32, device=self.device) for n in (nc, nt))
            # the tensor message channel (exchange_messages), per team: the episode id its totals belong to (-1 = restart
            # them at the next exchange) and the call serial that keys its dropout draws
            self._exchange_episode = tuple(torch.full((self.num_envs,), -1, dtype=torch.int32, device=self.device) for _ in range(2))
            self._exchange_serials = [0, 0]
        else:
            self._edges = (np.zeros((nc, nc), dtype=np.int64), np.zeros((nt, nt), dtype=np.int64))
            self._total_edges = (np.zeros((nc, nc), dtype=np.int64), np.zeros((nt, nt), dtype=np.int64))
        # the communication wrappers' combined rule per team (cameras, targets) for the batched greedy teams
        self.message_rules = {'range_limit': [np.inf, np.inf], 'keep_probability': [1.0, 1.0]}
        if self.batched:
            self.register_message_filter()

    # ------------------------------------------------------------------ configuration properties
    @property
    def unwrapped(self):
        return self

    @property
    def name(self) -> str:
        return self.config.get('name', 'MultiAgentTracking')

    num_cameras = property(lambda self: self.flat_config['num_cameras'])
    num_targets = property(lambda self: self.flat_config['num_targets'])
    num_obstacles = property(lambda self: self.flat_config['num_obstacles'])
    num_warehouses = property(lambda self: consts.NUM_WAREHOUSES)
    max_episode_steps = property(lambda self: self.flat_config['max_episode_steps'])
    camera_min_viewing_angle = property(lambda self: self.flat_config['camera_min_viewing_angle'])
    camera_max_sight_range = property(lambda self: self.flat_config['camera_max_sight_range'])
    camera_rotation_step = property(lambda self: self.flat_config['camera_rotation_step'])
    camera_zooming_step = property(lambda self: self.flat_config['camera_zooming_step'])
    target_step_size = property(lambda self: self.flat_config['target_step_size'])
    target_sight_range = property(lambda self: self.flat_config['target_sight_range'])
    num_cargoes_per_target = property(lambda self: self.flat_config['num_cargoes_per_target'])
    targets_start_with_cargoes = property(lambda self: bool(self.flat_config['targets_start_with_cargoes']))
    bounty_factor = property(lambda self: self.flat_config['bounty_factor'])
    obstacle_transmittance = property(lambda self: self.flat_config['obstacle_transmittance'])
    shuffle_entities = property(lambda self: bool(self.flat_config['shuffle_entities']))
    num_high_capacity_targets = property(lambda self: self.flat_config['num_high_capacity_targets'])
    num_low_capacity_targets = property(lambda self: self.num_targets - self.num_high_capacity_targets)
    camera_observation_dim = property(lambda self: self.sim.dc)
    target_observation_dim = property(lambda self: self.sim.dt)
    np_random = property(lambda self: self._np_random)

    def __str__(self) -> str:
        def plural(n, word):
            return f'{n} {word}{"s" if n > 1 else ""}'

        base = f'<{type(self).__name__} instance>' if self.spec is None else f'<{type(self).__name__}<{self.spec.id}>>'
        batch = f', {self.num_envs} envs' if self.batched else ''
        return (f'{base}({plural(self.num_cameras, "camera")}, {plural(self.num_targets, "target")}, '
                f'{plural(self.num_obstacles, "obstacle")}{batch})')

    # ------------------------------------------------------------------ core API
    def seed(self, seed: Optional[int] = None):
        """Key of the counter-based (Philox) reset / step streams (environment.py:1203-1227)."""
        if seed is None:
            seed = int(np.random.SeedSequence().entropy % (2 ** 63))
        self._seed = int(seed)
        self._np_random = np.random.RandomState(self._seed % (2 ** 32))
        self.sim.seed(self._seed % (2 ** 64))   # rewinds the episode counters: seed(s) + reset() is reproducible
        if self.batched:
            self._exchange_serials = [0, 0]       # and the message channel's drops
        return [self._seed]

    def load_config(self, config=None) -> None:
        """Re-initialise from another configuration, keeping wrappers (environment.py:564-588)."""
        seed = int(self._np_random.randint(2 ** 31 - 1))
        _, num_envs, device, base, _, observation_dtype, observed_team = self._init_args
        self.sim.close()
        self.__init__(config=config, num_envs=num_envs, device=device, env_index_base=base,  # pylint: disable=unnecessary-dunder-call
                      observation_dtype=observation_dtype, observed_team=observed_team)
        self.seed(seed)

    def reset(self, *, seed: Optional[int] = None):
        """Reset every environment; returns the first joint observation (environment.py:679-834)."""
        if seed is not None:
            self.seed(seed)
        cam_obs, tgt_obs = self.sim.reset()
        self.sim.observe(aux=True)   # refresh the mask attributes for the new episode
        self._needs_reset = False
        self._state_serial += 1
        if self.batched:   # environment.py:823-830
            for edges in self._delivered_bits + self._total_edges:
                edges.zero_()
            for episode in self._exchange_episode:
                episode.fill_(-1)
        else:
            for edges in self._edges + self._total_edges:
                edges.fill(0)
        self._clear_messages()
        return self._format_obs(cam_obs, tgt_obs)

    def _check_actions(self, action):
        camera_joint_action, target_joint_action = action
        nc, nt, B = self.num_cameras, self.num_targets, self.num_envs
        tgt = torch.as_tensor(np.asarray(target_joint_action) if not torch.is_tensor(target_joint_action) else target_joint_action,
                              dtype=torch.float32, device=self.device).reshape(B, nt, 2)
        if nc:
            cam = torch.as_tensor(np.asarray(camera_joint_action) if not torch.is_tensor(camera_joint_action) else camera_joint_action,
                                  dtype=torch.float32, device=self.device).reshape(B, nc, 2)
        else:
            cam = None
        if not self.batched or getattr(self, 'check_finite', False):
            # the reference asserts finiteness (environment.py:1337-1342); in batched mode the check
            # costs a device sync, so it is opt-in via `env.check_finite = True`
            if (cam is not None and not bool(torch.isfinite(cam).all())) or not bool(torch.isfinite(tgt).all()):
                raise AssertionError(f'Got unexpected joint action {action}.')
        return cam, tgt

    def step(self, action):
        """Run one timestep for every environment (environment.py:590-676)."""
        if self._needs_reset:
            raise RuntimeError('call reset() before step()')
        cam, tgt = self._check_actions(action)
        # parity hook: `env.replay_next = (transmit, goal_choice)` replays recorded draws of the reference in this step
        replay = self.__dict__.pop('replay_next', None)
        (cam_obs, tgt_obs), rewards, done = self.sim.step(cam, tgt, auto_reset=self.batched, aux=True, replay=replay)
        self._step_serial += 1
        self._state_serial += 1
        if self.batched:
            aux = self._aux
            common = {
                'coverage_rate': aux['coverage'][:, 0], 'real_coverage_rate': aux['coverage'][:, 1],
                'mean_transport_rate': aux['coverage'][:, 2], 'num_delivered_cargoes': aux['num_delivered'],
                'episode_step': aux['episode_step'],
            }
            scale = 1.0 / self.max_target_team_episode_reward
            camera_infos = dict(common, raw_reward=rewards[:, 0], normalized_raw_reward=rewards[:, 0] * scale)
            target_infos = dict(common, raw_reward=rewards[:, 1], normalized_raw_reward=rewards[:, 1] * scale,
                                target_dones=aux['target_dones'], is_colliding=aux['is_colliding'])
            return (cam_obs, tgt_obs), (rewards[:, 0], rewards[:, 1]), done.bool(), (camera_infos, target_infos)
        # ---- reference-compatible single-env return types ----
        rew = rewards[0].tolist()
        done_flag = bool(done[0].item())
        cov = self._aux['coverage'][0].tolist()
        common = {
            'coverage_rate': cov[0], 'real_coverage_rate': cov[1], 'mean_transport_rate': cov[2],
            'num_delivered_cargoes': int(self._aux['num_delivered'][0].item()),
        }
        norm = self.max_target_team_episode_reward
        # the messages sent since the previous step reach their recipients through the infos (environment.py:641-669)
        cam_edges, tgt_edges = self.communication_edges
        camera_infos = [dict(raw_reward=rew[0], normalized_raw_reward=rew[0] / norm, messages=self.camera_message_buffer[c],
                             out_communication_edges=cam_edges[c, :].sum(), in_communication_edges=cam_edges[:, c].sum(), **common)
                        for c in range(self.num_cameras)]
        target_infos = [dict(raw_reward=rew[1], normalized_raw_reward=rew[1] / norm, messages=self.target_message_buffer[t],
                             out_communication_edges=tgt_edges[t, :].sum(), in_communication_edges=tgt_edges[:, t].sum(), **common)
                        for t in range(self.num_targets)]
        for total, edges in zip(self.total_communication_edges, self.communication_edges):
            total += edges
            edges.fill(0)
        self._clear_messages()
        return self._format_obs(cam_obs, tgt_obs), (rew[0], rew[1]), done_flag, (camera_infos, target_infos)

    # ------------------------------------------------------------------ communication edges and filter
    def register_message_filter(self):
        """Register ``message_rules`` and, in batched mode, the edge tensors with the simulator: the batched greedy
        teams of ``MultiCamera`` / ``MultiTarget`` apply the rules to the messages they exchange inside their kernels
        and count what is delivered.  Teams of more than 8 agents are not counted (the bit matrix holds 8)."""
        nc, nt = self.num_cameras, self.num_targets
        counted = [self.batched and 0 < n <= 8 for n in (nc, nt)]
        self.sim.set_message_filter(
            range_limit=tuple(self.message_rules['range_limit']), keep_probability=tuple(self.message_rules['keep_probability']),
            delivered=tuple(self._delivered_bits[t] if counted[t] else None for t in range(2)),
            total_edges=tuple(self._total_edges[t] if counted[t] else None for t in range(2)))

    @staticmethod
    def _unpack_edges(bits, n):
        shift = 8 * torch.arange(n, device=bits.device).view(n, 1) + torch.arange(n, device=bits.device).view(1, n)
        return ((bits.view(-1, 1, 1) >> shift) & 1).bool()

    @property
    def communication_edges(self):
        """Per team (cameras, targets): messages delivered since the last step.  Batched: ``[B, N, N]`` bool, the
        delivered set of the greedy team's last call, sender-major; single environment: the reference's NumPy counts of
        the host ``Message`` traffic."""
        if self.batched:
            return tuple(self._unpack_edges(bits, n) for bits, n in zip(self._delivered_bits, (self.num_cameras, self.num_targets)))
        return self._edges

    @property
    def total_communication_edges(self):
        """Per team: messages delivered in the episode.  Batched: ``[B, N, N]`` int32, since the environment's greedy
        agents were last reset; single environment: NumPy, since ``reset``."""
        return self._total_edges

    camera_communication_edges = property(lambda self: self.communication_edges[0])
    target_communication_edges = property(lambda self: self.communication_edges[1])
    camera_total_communication_edges = property(lambda self: self._total_edges[0])
    target_total_communication_edges = property(lambda self: self._total_edges[1])

    # ------------------------------------------------------------------ tensor messages of a learning team (batched mode)
    def exchange_messages(self, team, content, recipients=None, reduction: str = 'none'):
        """Send one message per agent of ``team`` (``'camera'`` / ``'target'``, 0 / 1 or ``Team``) and receive them, for
        every environment in one kernel (DESIGN.md section 7i).  ``content`` float32 ``[B, N, D]`` on the environment's
        device; ``recipients`` bool / uint8 ``[B, N, N]`` sender-major (entry ``[e, s, r]``: s sends to r), ``None`` =
        broadcast to every teammate, the sender included.  A message is delivered iff it is sent and passes the
        communication wrappers registered for the team (range on the current positions, dropout).  Returns ``(inbox,
        delivered)``: ``inbox`` float32 ``[B, N(r), N(s), D]`` with s's message where it reached r and zeros elsewhere
        (``reduction='none'``), or ``[B, N(r), D]``, the sum / mean over the delivered senders (``'sum'`` / ``'mean'``,
        0 without any); ``delivered`` bool ``[B, N(r), N(s)]``.  The delivered set also becomes the team's
        ``communication_edges`` and is added to its ``total_communication_edges``, which restart at the first exchange of
        an episode."""
        if not self.batched:
            raise NotImplementedError('exchange_messages is the message channel of the batched mode (num_envs=B); the '
                                      'single-environment mode exchanges Message objects with send_messages / receive_messages')
        try:
            index = consts._team_index(team)   # pylint: disable=protected-access
        except (KeyError, TypeError, ValueError):
            index = None
        if index not in (0, 1):
            raise ValueError(f"team must be 'camera' / 'target', 0 / 1 or a Team, got {team!r}")
        out = self.sim.exchange_messages(index, content, recipients, reduction, self._exchange_serials[index], self._exchange_episode[index])
        self._exchange_serials[index] += 1
        return out

    # ------------------------------------------------------------------ intra-team messages (reference-compatible mode)
    def _clear_messages(self):
        for table in self.message_buffers + self.message_queues:
            table.clear()

    def _messages_supported(self):
        if self.batched:
            raise NotImplementedError(
                'Message objects are a host API of the single-environment mode (num_envs=None); in batched mode learning '
                'teams exchange tensor messages with exchange_messages, and the greedy teams exchange theirs inside '
                'their CUDA kernels (mate_b200.MultiCamera / MultiTarget)')

    def send_messages(self, messages) -> None:
        """Buffer messages from an agent to teammates; they are delivered by ``receive_messages`` and through the
        ``'messages'`` entry of the next step's infos (mate/environment.py:836-854).  Accepts the reference's
        ``mate.utils.Message`` objects as well as ``mate_b200.Message``."""
        self._messages_supported()
        if hasattr(messages, 'sender') and hasattr(messages, 'content'):
            messages = (messages,)
        messages = list(messages)
        assert len({consts._team_index(m.team) for m in messages}) <= 1, (   # pylint: disable=protected-access
            f'All messages must be from the same team. Got messages = {messages}.')
        for message in self.route_messages(messages):
            team = consts._team_index(message.team)   # pylint: disable=protected-access
            self.message_queues[team][message.recipient].append(message)
            self.message_buffers[team][message.recipient].append(message)
            self.communication_edges[team][message.sender, message.recipient] += 1

    def receive_messages(self, agent_id=None, agent=None):
        """Messages waiting for one agent (``agent_id = (team, index)`` or an agent object with ``TEAM`` and
        ``index``) or, without arguments, for all agents of both teams (mate/environment.py:856-892)."""
        self._messages_supported()
        if agent_id is None and agent is None:
            messages = ([list(self.camera_message_queue[c]) for c in range(self.num_cameras)],
                        [list(self.target_message_queue[t]) for t in range(self.num_targets)])
            self.camera_message_queue.clear()
            self.target_message_queue.clear()
            return messages
        if agent is None and hasattr(agent_id, 'TEAM') and hasattr(agent_id, 'index'):
            agent_id, agent = None, agent_id
        if agent is not None:
            assert agent_id is None, ('You should specify either `agent_id` or `agent`, not both.'
                                      f'Got (agent_id, agent) = {(agent_id, agent)}.')
            team, index = agent.TEAM, agent.index
        else:
            team, index = agent_id
        queue = self.message_queues[consts._team_index(team)]   # pylint: disable=protected-access
        messages = list(queue[index])
        del queue[index]
        return messages

    def route_messages(self, messages):
        """Broadcast messages (``recipient is None``) become one peer-to-peer copy per teammate, the sender included
        (mate/environment.py:1249-1269)."""
        routed = []
        for message in messages:
            if message.recipient is None:
                num_teammates = (self.num_cameras, self.num_targets)[consts._team_index(message.team)]   # pylint: disable=protected-access
                for recipient in range(num_teammates):
                    routed.append(type(message)(sender=message.sender, recipient=recipient, content=copy.deepcopy(message.content),
                                                team=message.team, broadcasting=True))
            else:
                routed.append(message)
        return routed

    def add_render_callback(self, name: str, callback) -> None:
        """Kept for wrappers that register one (mate/environment.py:1181-1186); never called: the callbacks draw pyglet
        geometry, and ``render`` draws its frames on the GPU."""
        self.render_callbacks[name] = callback

    def joint_observation(self):
        """Joint observations of both teams for the current state (environment.py:908-983); ``None`` for a team that is
        not observed (``observed_team``)."""
        cam_obs, tgt_obs = self.sim.observe(aux=True)
        return self._format_obs(cam_obs, tgt_obs)

    def _format_obs(self, cam_obs, tgt_obs):
        if self.batched:
            return cam_obs, tgt_obs
        return cam_obs[0].double().cpu().numpy(), tgt_obs[0].double().cpu().numpy()

    def _maybe_single(self, array):
        return array if self.batched else array[0]

    # ------------------------------------------------------------------ state access
    def get_state(self) -> Dict[str, np.ndarray]:
        """A view of the simulator state as host arrays (fields of ``MateStateView``).  It is not a complete checkpoint
        (the running coverage sum, the line-of-sight cache, the seed and the episode statistics are left out):
        ``save_state`` / ``load_state`` save and restore a batch exactly."""
        return self.sim.get_state()

    def save_state(self, envs=None):
        """Snapshot of the environments ``envs`` (``None`` = all; entry i = environment ``envs[i]``) on the device, with
        this object's seed and NumPy RNG state (a :class:`mate_b200.sim.StateSnapshot`; ``torch.save`` keeps it)."""
        snapshot = self.sim.save_state(envs)
        kind, key, pos, has_gauss, cached = self._np_random.get_state()
        saved = {'seed': self._seed, 'np_random': (kind, torch.from_numpy(key.astype(np.int64)), pos, has_gauss, cached)}
        if self.batched:   # both teams' communication totals and the message channel's bookkeeping
            index = None
            if envs is not None:   # out-of-range device indices: the kernel leaves those entries unwritten, here they are clamped
                index = self.sim._index_map(envs, 'envs', None, 0, self.num_envs).long().clamp_(0, self.num_envs - 1)  # pylint: disable=protected-access
            pick = lambda t: (t if index is None else t.index_select(0, index)).clone()   # noqa: E731
            saved.update(total_edges=tuple(pick(t) for t in self._total_edges),
                         exchange_episode=tuple(pick(t) for t in self._exchange_episode),
                         exchange_serials=list(self._exchange_serials))
        snapshot.extras['environment'] = saved
        return snapshot

    def load_state(self, snapshot, src=None, resume: bool = False):
        """Load a snapshot and return the joint observation of the loaded state, like ``reset``.  ``src=None``: every
        environment takes its own entry; otherwise environment d takes entry ``src[d]`` (a negative entry keeps d), e.g.
        ``env.load_state(env.save_state(), src=idx)`` branches the batch from the environments ``idx``.  ``resume=True``
        continues exactly where the snapshot was saved: it also restores the seed, the episode statistics and the NumPy
        RNG state."""
        self.sim.load_state(snapshot, src=src, resume=resume)
        saved = snapshot.extras.get('environment')
        if resume and saved is not None:
            kind, key, pos, has_gauss, cached = saved['np_random']
            self._seed = saved['seed']
            self._np_random.set_state((kind, key.numpy().astype(np.uint32), pos, has_gauss, cached))
        if self.batched and saved is not None and 'total_edges' in saved:   # older snapshots do not carry them
            self._load_rows(self._total_edges + self._exchange_episode, saved['total_edges'] + saved['exchange_episode'],
                            src, snapshot.count)
            if resume:
                self._exchange_serials = list(saved['exchange_serials'])
        cam_obs, tgt_obs = self.sim.observe(aux=True)   # the mask attributes of the loaded state
        self._needs_reset = False
        self._state_serial += 1
        return self._format_obs(cam_obs, tgt_obs)

    def _load_rows(self, live, saved, src, count):
        """Per-environment tensors (environment axis first) from a snapshot's entries along its index map, with the
        simulator's rules: ``src=None`` takes entry d for environment d, a negative or out-of-range entry keeps d."""
        index = None
        if src is not None:
            index = self.sim._index_map(src, 'src', self.num_envs, -(1 << 31), count).long()  # pylint: disable=protected-access
            keep = (index < 0) | (index >= count)
            index = index.clamp(0, count - 1)
        for tensor, rows in zip(live, saved):
            rows = rows.to(tensor.device)
            if index is None:
                tensor.copy_(rows)
            else:
                tensor.copy_(torch.where(keep.view((-1,) + (1,) * (tensor.dim() - 1)), tensor, rows.index_select(0, index)))

    def set_state(self, arrays: Dict[str, np.ndarray]) -> None:
        """Inject a state (the reference has no equivalent; used by the parity harness).  For checkpoint / resume use
        ``save_state`` / ``load_state``."""
        self.sim.set_state(arrays)
        if self.batched:   # the message channel's totals restart at the next exchange
            for episode in self._exchange_episode:
                episode.fill_(-1)
        self.sim.observe(aux=True)
        self._needs_reset = False
        self._state_serial += 1

    def state(self) -> np.ndarray:
        """The global state vector (environment.py:894-906), ``[B, D]`` float64 (``[D]`` in
        reference-compatible mode)."""
        s = self.sim.get_state()
        B, nc, nt, no = self.num_envs, self.num_cameras, self.num_targets, self.num_obstacles
        cfg = self.flat_config
        preserved = np.concatenate([[nc, nt, no, 0.0], consts.WAREHOUSES.ravel(), [consts.WAREHOUSE_RADIUS]])
        rs = np.sqrt(cfg['camera_min_viewing_angle'] * cfg['camera_max_sight_range'] ** 2 / s['cam_theta']) if nc else np.zeros((B, 0))
        phi = np.deg2rad(s['cam_phi'])
        cam = np.stack([
            s['cam_xy'][..., 0], s['cam_xy'][..., 1], np.full((B, nc), cfg['camera_radius']),
            rs * np.cos(phi), rs * np.sin(phi), s['cam_theta'], np.full((B, nc), cfg['camera_max_sight_range']),
            np.full((B, nc), cfg['camera_rotation_step']), np.full((B, nc), cfg['camera_zooming_step']),
        ], axis=-1).reshape(B, nc * 9)
        goal_bits = np.zeros((B, nt, 4))
        has_goal = s['tgt_goal'] >= 0
        b_idx, t_idx = np.nonzero(has_goal)
        goal_bits[b_idx, t_idx, s['tgt_goal'][has_goal]] = s['tgt_weight'][has_goal]
        empty = (s['tgt_empty_bits'][..., None] >> np.arange(4)) & 1
        tgt = np.concatenate([
            s['tgt_xy'], np.full((B, nt, 1), cfg['target_sight_range']), (goal_bits.sum(-1, keepdims=True) > 0),
            (cfg['target_step_size'] / s['tgt_capacity'])[..., None], s['tgt_capacity'][..., None], goal_bits, empty,
        ], axis=-1).reshape(B, nt * 14)
        freights = s['tgt_weight'] * self.freight_scale
        out = np.concatenate([np.tile(preserved, (B, 1)), cam, tgt, s['obs_xyr'].reshape(B, no * 3), freights,
                              s['tgt_bounty'], s['remaining'].reshape(B, 16)], axis=-1).astype(np.float64)
        return self._maybe_single(out)

    # ------------------------------------------------------------------ attributes wrappers and agents read
    def _snapshot(self):
        """Host copy of the simulator state, taken once per step / reset / set_state on first use: the entity
        views and the cargo attributes below all read the same snapshot."""
        serial, snap = self._snapshot_cache
        if serial != self._state_serial:
            snap = self.sim.get_state()
            self._snapshot_cache = (self._state_serial, snap)
        return snap

    def _aux_numpy(self, key):
        return self._aux[key].cpu().numpy()

    def _host(self, tensor, dtype=None):
        """A per-step device tensor in the type of the calling convention: the tensor itself (``[B, ...]``) in
        batched mode, a NumPy array without the batch dimension in reference-compatible mode."""
        if self.batched:
            return tensor if dtype is not bool else tensor.bool()
        out = tensor[0].cpu().numpy()
        return out.astype(dtype) if dtype is not None else out

    # view masks (mate/environment.py:475-495)
    camera_target_view_mask = property(lambda self: self._host(self._aux['mask_ct'], bool))
    camera_camera_view_mask = property(lambda self: self._host(self._aux['mask_cc'], bool))
    camera_obstacle_view_mask = property(lambda self: self._host(self._aux['mask_co'], bool))
    target_camera_view_mask = property(lambda self: self._host(self._aux['mask_tc'], bool))
    target_obstacle_view_mask = property(lambda self: self._host(self._aux['mask_to'], bool))
    target_target_view_mask = property(lambda self: self._host(self._aux['mask_tt'], bool))
    target_dones = property(lambda self: self._host(self._aux['target_dones'], bool))
    target_warehouse_distances = property(lambda self: self._host(self._aux['warehouse_dist'], np.float64))

    @property
    def tracked_bits(self):
        """camera_target_view_mask.any(axis=0) (mate/environment.py:1387)."""
        mask = self.camera_target_view_mask
        return mask.any(dim=1) if self.batched else mask.any(axis=0)

    def _scalar(self, tensor, cast):
        return tensor if self.batched else cast(tensor[0].item())

    coverage_rate = property(lambda self: self._scalar(self._aux['coverage'][:, 0], float))
    real_coverage_rate = property(lambda self: self._scalar(self._aux['coverage'][:, 1], float))
    mean_transport_rate = property(lambda self: self._scalar(self._aux['coverage'][:, 2], float))
    num_delivered_cargoes = property(lambda self: self._scalar(self._aux['num_delivered'], int))
    episode_step = property(lambda self: self._scalar(self._aux['episode_step'], int))
    # cargo tables and per-target integers (mate/environment.py:503-519): from the host snapshot
    remaining_cargoes = property(lambda self: self._maybe_single(self._snapshot()['remaining'].astype(np.int64)))
    awaiting_cargo_counts = property(lambda self: self._maybe_single(self._snapshot()['awaiting'].astype(np.int64)))
    target_goals = property(lambda self: self._maybe_single(self._snapshot()['tgt_goal'].astype(np.int64)))
    target_capacities = property(lambda self: self._maybe_single(self._snapshot()['tgt_capacity'].astype(np.int64)))
    target_team_episode_reward = property(lambda self: self._maybe_single(self._snapshot()['episode_reward'][:, 0]))
    delayed_target_team_episode_reward = property(lambda self: self._maybe_single(self._snapshot()['episode_reward'][:, 1]))
    obstacle_states = property(lambda self: self._maybe_single(self._snapshot()['obs_xyr'].astype(np.float64)))

    @property
    def target_goal_bits(self):
        """[Nt, 4]: the cargo weight at the index of each target's goal warehouse (mate/environment.py:1305-1309)."""
        snap = self._snapshot()
        bits = (np.arange(consts.NUM_WAREHOUSES) == snap['tgt_goal'][..., None]) * snap['tgt_weight'][..., None]
        return self._maybe_single(bits.astype(np.int64))

    @property
    def obstacle_states_flagged(self):
        """Obstacle states with a trailing 1 (mate/environment.py:471, 747-750)."""
        states = self._snapshot()['obs_xyr'].astype(np.float64)
        return self._maybe_single(np.concatenate([states, np.ones(states.shape[:-1] + (1,))], axis=-1))

    @property
    def camera_obstacle_observations(self):
        """Per camera, the flagged obstacle states masked by its obstacle set, flattened (mate/environment.py:757-764)."""
        flagged = self._snapshot()['obs_xyr'].astype(np.float64)
        flagged = np.concatenate([flagged, np.ones(flagged.shape[:-1] + (1,))], axis=-1)            # [B, No, 4]
        mask = self._aux_numpy('mask_co').astype(bool)                                              # [B, Nc, No]
        out = np.where(mask[..., None], flagged[:, None], 0.0).reshape(self.num_envs, self.num_cameras, -1)
        return self._maybe_single(out)

    target_goals_of_last_step = property(lambda self: self._maybe_single(self._aux['tgt_goal']))

    def auxiliary_terms(self):
        """``(cam_terms [B, Nc, 8], tgt_terms [B, Nt, 16])`` of the last step, computed once per step by one kernel
        and shared by the auxiliary-reward / training-information wrappers (``include/mate_b200.h``,
        ``mate_b200_auxiliary_terms``)."""
        if self._terms_serial != self._step_serial:
            soft = self.sim.soft_coverage(auto_reset=self.batched) if (self.want_soft_coverage and self.num_cameras) else None
            self._terms = self.sim.auxiliary_terms(soft)
            self._terms_serial = self._step_serial
        return self._terms

    def episode_statistics(self, reduce_across_ranks: bool = False, reset: bool = False) -> Dict[str, float]:
        """Episode statistics accumulated on the device; with ``reduce_across_ranks`` the
        16-float vector is all-reduced over the process group (NCCL) -- the only collective
        of the whole simulator, and never on the step path."""
        stats = self.sim.episode_stats(reset_after=reset).clone()
        if reduce_across_ranks:
            import torch.distributed as dist  # pylint: disable=import-outside-toplevel

            if dist.is_available() and dist.is_initialized():
                dist.all_reduce(stats, op=dist.ReduceOp.SUM)
        values = stats.cpu().tolist()
        episodes = max(values[0], 1.0)
        return {
            'episodes': values[0], 'mean_return': values[1] / episodes, 'mean_length': values[2] / episodes,
            'mean_delivered': values[3] / episodes, 'mean_coverage': values[4] / episodes, 'env_steps': values[5],
        }

    def render(self, mode='human', window_size=800, envs=None):
        """An ``rgb_array`` frame of the current state, drawn on the GPU (DESIGN.md section 7k): the terrain, warehouses,
        the cameras' fields of view (darker where several cameras overlap), obstacles, cameras and targets (filled with
        the goal warehouse's colour when loaded, ringed when tracked).  Single environment: NumPy uint8
        ``[window_size, window_size, 3]``, the reference's type.  Batched: a CUDA uint8 tensor ``[K, S, S, 3]`` of the
        environments ``envs`` (default: environment 0 only), written on the current stream.  ``mode='human'`` (a
        window) is not supported.  The registered ``render_callbacks`` are kept but never called: they draw pyglet
        geometry."""
        if mode != 'rgb_array':
            raise NotImplementedError(f"render mode {mode!r} is not supported: this environment has no window; use "
                                      "render(mode='rgb_array') for frames")
        if self._needs_reset:
            raise RuntimeError('call reset() before render()')
        if not self.batched and envs is not None:
            raise ValueError('envs applies to the batched mode (num_envs=B)')
        check_render_size(window_size)
        envs = [0] if envs is None else envs
        check_index_map(envs, 'envs', None, 0, self.num_envs)
        frames = self.sim.render(envs, size=window_size)
        return frames if self.batched else frames[0].cpu().numpy()

    def close(self) -> None:
        self.sim.close()
