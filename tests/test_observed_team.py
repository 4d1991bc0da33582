"""Observation rows for one team (``observed_team='camera' | 'target'``, NULL row pointers in the C ABI): the step kernel
composes and writes only the observed team's rows, and everything else -- the observed rows, rewards, done, every
auxiliary output, the state and the snapshots -- is bit for bit what a both-teams simulator computes on the same seed
and actions."""

import ctypes
import gc
import os

import numpy as np
import pytest

torch = pytest.importorskip('torch')

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
PRESETS = [f'MATE-{nc}v{nt}-{no}.yaml' for nc, nt in ((1, 1), (1, 2), (2, 2), (2, 4), (4, 2), (4, 4), (4, 8), (8, 8))
           for no in (0, 9)] + ['MATE-Navigation.yaml']
CASES = [(preset, team) for preset in PRESETS for team in ('camera', 'target') if not (preset == 'MATE-Navigation.yaml' and team == 'camera')]


# ---------------------------------------------------------------------------------------------- CPU
def test_observed_team_is_checked_before_anything_is_allocated():
    from mate_b200.config import flatten_config, read_config
    from mate_b200.environment import MultiAgentTracking
    from mate_b200.sim import BatchedSim

    cfg = flatten_config(read_config('MATE-4v8-9.yaml'))
    nav = flatten_config(read_config('MATE-Navigation.yaml'))
    for team in ('cameras', 'none', None, 0, 'Both'):
        with pytest.raises(ValueError, match='observed_team'):
            BatchedSim(cfg, 16, observed_team=team)
        with pytest.raises(ValueError, match='observed_team'):
            MultiAgentTracking('MATE-4v8-9.yaml', num_envs=16, observed_team=team)
    with pytest.raises(ValueError, match='cameras'):
        BatchedSim(nav, 16, observed_team='camera')
    with pytest.raises(ValueError, match='cameras'):
        MultiAgentTracking('MATE-Navigation.yaml', num_envs=16, observed_team='camera')
    for team in ('camera', 'target'):   # the single-environment mode returns both teams' NumPy rows
        with pytest.raises(ValueError, match='batched'):
            MultiAgentTracking('MATE-4v8-9.yaml', observed_team=team)


def _recorded_env(observed_team):
    """A batched environment of one environment over the recorded observations of wrappers_4v8-9.npz, with a simulator
    that takes ``observed_team`` like BatchedSim (None for the team it does not observe)."""
    import mate_b200.environment as b200
    from test_communication_wrappers import FilterRecordingSim

    g = np.load(os.path.join(GOLDEN, 'wrappers_4v8-9.npz'))
    base = FilterRecordingSim.make()
    seen = []

    class Sim(base):
        fixture = (g, 'w_')

        def __init__(self, flat_config, num_envs, device=0, env_index_base=0, **kwargs):
            seen.append(dict(kwargs))
            super().__init__(flat_config, num_envs, device=device, env_index_base=env_index_base)
            self.observed_team = kwargs.get('observed_team', 'both')
            self.cam_obs = None if self.observed_team == 'target' else torch.zeros((1, self.nc, self.dc))

        def _drop(self, rows):
            cam, tgt = rows
            return (None if self.observed_team == 'target' else cam, None if self.observed_team == 'camera' else tgt)

        def observe(self, replay=None, aux=False):
            return self._drop(super().observe(replay=replay, aux=aux))

        def step(self, cam_act, tgt_act, auto_reset=True, replay=None, aux=False):
            rows, rewards, done = super().step(cam_act, tgt_act, auto_reset=auto_reset, replay=replay, aux=aux)
            return self._drop(rows), rewards, done

    env = type('MultiAgentTracking', (b200.MultiAgentTracking,), {'_sim_class': Sim})(
        config=str(g['config_name']), num_envs=1, observed_team=observed_team)
    return env, seen


@pytest.mark.parametrize('team', ['both', 'camera', 'target'])
def test_joint_observations_hold_none_for_the_team_not_observed(team):
    env, seen = _recorded_env(team)
    assert seen == [{} if team == 'both' else {'observed_team': team}]   # the default is not passed on
    slot = {'both': None, 'camera': 1, 'target': 0}[team]

    def check(joint):
        assert len(joint) == 2
        for k in range(2):
            assert (joint[k] is None) == (k == slot), (team, k)

    check(env.reset())
    nc, nt = env.num_cameras, env.num_targets
    joint, _, _, _ = env.step((torch.zeros((1, nc, 2)), torch.zeros((1, nt, 2))))
    check(joint)
    check(env.joint_observation())
    assert env.observation_space.spaces[0].spaces[0].shape == (env.camera_observation_dim,)   # spaces and dims stay
    assert env.target_observation_dim == env.sim.dt
    env.load_config()
    assert env.observed_team == team and seen[-1] == seen[0]
    import mate_b200

    if team != 'both':   # a single-team wrapper needs its learning team's rows, MultiTarget the camera rows as well
        with pytest.raises(ValueError, match='camera rows'):
            mate_b200.MultiTarget(env, camera_agent=mate_b200.GreedyCameraAgent(seed=0))
    if team == 'target':
        with pytest.raises(ValueError, match='MultiCamera returns the camera rows'):
            mate_b200.MultiCamera(env, target_agent=mate_b200.GreedyTargetAgent(seed=0))


@pytest.mark.parametrize('team', ['both', 'camera', 'target'])
def test_step_host_refuses_buffers_that_do_not_fit_the_observed_team(team):
    """BatchedSim.step_host checks the row buffers against observed_team before the library call: a buffer for a team
    that is not observed, or None for one that is, raises ValueError."""
    from mate_b200.sim import BatchedSim

    class NoLibrary:
        def __getattr__(self, name):
            raise AssertionError(f'the library was called ({name}) although the arguments are refused')

    B, nc, nt, dc, dt = 4, 4, 8, 126, 131
    sim = BatchedSim.__new__(BatchedSim)   # the host-side checks only: no device, no handle
    sim.lib, sim.handle, sim.nc, sim.observed_team, sim.observation_dtype = NoLibrary(), None, nc, team, torch.float32
    sim.cam_obs = None if team == 'target' else torch.zeros((B, nc, dc))
    sim.tgt_obs = None if team == 'camera' else torch.zeros((B, nt, dt))
    cam_rows, tgt_rows = torch.zeros((B, nc, dc)), torch.zeros((B, nt, dt))
    rewards, done = torch.zeros((B, 2)), torch.zeros(B, dtype=torch.uint8)
    act = (torch.zeros((B, nc, 2)), torch.zeros((B, nt, 2)))
    for cam, tgt in ((None, tgt_rows), (cam_rows, None), (None, None), (cam_rows, tgt_rows)):
        fits = (cam is not None) == (team != 'target') and (tgt is not None) == (team != 'camera')
        if not fits:
            with pytest.raises(ValueError, match='step_host'):
                sim.step_host(*act, (cam, tgt, rewards, done))
        else:
            with pytest.raises(AssertionError, match='library was called'):   # the checks let it through
                sim.step_host(*act, (cam, tgt, rewards, done))


# ---------------------------------------------------------------------------------------------- GPU
def _sims(preset, B, team, dtype=torch.float32, **overrides):
    from mate_b200.config import flatten_config, read_config
    from mate_b200.sim import BatchedSim

    cfg = flatten_config(read_config(preset, **overrides))
    return cfg, BatchedSim(cfg, B, device=0, observation_dtype=dtype), BatchedSim(cfg, B, device=0, observation_dtype=dtype, observed_team=team)


def _actions(cfg, B, k):
    gen = torch.Generator(device='cuda')
    gen.manual_seed(2000 + k)
    scale = torch.tensor([cfg['camera_rotation_step'], cfg['camera_zooming_step']], device='cuda')
    cam = (torch.rand((B, max(cfg['num_cameras'], 1), 2), device='cuda', generator=gen) * 2 - 1) * scale
    tgt = (torch.rand((B, cfg['num_targets'], 2), device='cuda', generator=gen) * 2 - 1) * cfg['target_step_size']
    return cam[:, :cfg['num_cameras']].contiguous(), tgt


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.float16 else t.view(torch.int32)


def _same_snapshots(a, b):
    """Equal snapshot payloads but for the floating-point sums among the episode statistics at their end (float atomics,
    added in no fixed order); the counters there are compared."""
    pa, pb = a.save_state().payload, b.save_state().payload
    sa, sb = pa[-64:].view(torch.float32), pb[-64:].view(torch.float32)
    exact = [0, 1, 2, 3, 5]   # episodes, rewards, steps, deliveries (integers in float32), env-steps
    return torch.equal(pa[:-64], pb[:-64]) and torch.equal(sa[exact], sb[exact])


def _assert_same(both, one, ctx, aux=True, snapshot=True):
    """``one`` observes a single team: its rows equal ``both``'s rows of that team, the other tensor is None, and
    rewards, done, aux and the saved state are identical."""
    torch.cuda.synchronize()
    for mine, ref, name in ((one.cam_obs, both.cam_obs, 'cam_obs'), (one.tgt_obs, both.tgt_obs, 'tgt_obs')):
        observed = one.observed_team in ('both', 'camera' if name == 'cam_obs' else 'target')
        if observed:
            assert torch.equal(_bits(mine), _bits(ref)), (ctx, name)
        else:
            assert mine is None, (ctx, name)
    assert torch.equal(one.rewards, both.rewards) and torch.equal(one.done, both.done), ctx
    if aux:
        for key, value in both.aux.items():
            assert torch.equal(value, one.aux[key]), (ctx, key)
    if snapshot:
        assert _same_snapshots(one, both), (ctx, 'snapshot')


@pytest.mark.gpu
@pytest.mark.parametrize('refill', ['sync', 'default'])
@pytest.mark.parametrize('preset,team', CASES)
def test_every_preset_and_team_matches_both(preset, team, refill, monkeypatch):
    """A ragged batch with episodes short enough that most environments auto-reset, float32 and float16 rows."""
    if refill == 'sync':
        monkeypatch.setenv('MATE_B200_REFILL', 'sync')
    else:
        monkeypatch.delenv('MATE_B200_REFILL', raising=False)
    B = 1001
    for dtype in (torch.float32, torch.float16):
        cfg, both, one = _sims(preset, B, team, dtype, max_episode_steps=4)
        both.reset(seed=11)
        one.reset(seed=11)
        _assert_same(both, one, (preset, team, dtype, 'reset'), aux=False)
        for k in range(11):
            cam, tgt = _actions(cfg, B, k)
            both.step(cam, tgt, auto_reset=True, aux=True)
            one.step(cam, tgt, auto_reset=True, aux=True)
            _assert_same(both, one, (preset, team, dtype, k), snapshot=(k % 3 == 2))
        assert int(one.episode_stats()[0]) >= B   # the auto-reset paths ran
        assert torch.equal(one.episode_stats()[[0, 1, 2, 3, 5]], both.episode_stats()[[0, 1, 2, 3, 5]])
        both.close()
        one.close()


@pytest.mark.gpu
@pytest.mark.parametrize('tile', ['32', '16', '8'])
def test_full_size_4v8_9(tile, monkeypatch):
    """MATE-4v8-9 x 65 536 with the asynchronous refill and every warp tile size, both single teams."""
    monkeypatch.setenv('MATE_B200_TILE', tile)
    monkeypatch.delenv('MATE_B200_REFILL', raising=False)
    from mate_b200.sim import BatchedSim

    B = 65536
    cfg, both, cams = _sims('MATE-4v8-9.yaml', B, 'camera', max_episode_steps=5)
    tgts = BatchedSim(cfg, B, device=0, observed_team='target')
    for sim in (both, cams, tgts):
        sim.reset(seed=2)
    for k in range(8):
        cam, tgt = _actions(cfg, B, k)
        for sim in (both, cams, tgts):
            sim.step(cam, tgt, auto_reset=True, aux=True)
        _assert_same(both, cams, ('full', tile, 'camera', k), snapshot=(k == 7))
        _assert_same(both, tgts, ('full', tile, 'target', k), snapshot=(k == 7))
    for sim in (both, cams, tgts):
        sim.close()


@pytest.mark.gpu
@pytest.mark.parametrize('team', ['camera', 'target'])
@pytest.mark.parametrize('preset', ['MATE-4v8-9.yaml', 'MATE-4v2-9.yaml', 'MATE-8v8-9.yaml'])
def test_masked_reset_observe_after_set_state_and_branching(preset, team, monkeypatch):
    monkeypatch.setenv('MATE_B200_REFILL', 'sync')
    B = 300
    cfg, both, one = _sims(preset, B, team, max_episode_steps=6)
    both.reset(seed=5)
    one.reset(seed=5)
    for k in range(4):
        cam, tgt = _actions(cfg, B, k)
        both.step(cam, tgt, aux=True)
        one.step(cam, tgt, aux=True)
    rng = np.random.RandomState(4)
    mask = torch.from_numpy(rng.randint(0, 2, B).astype(np.uint8)).cuda()
    both.reset(env_mask=mask)
    one.reset(env_mask=mask)
    _assert_same(both, one, (preset, team, 'masked reset'), aux=False)
    state = both.get_state()
    for sim in (both, one):
        sim.set_state(state)
        sim.observe(aux=True)
    _assert_same(both, one, (preset, team, 'observe after set_state'))
    assert _same_snapshots(both, one)
    snap_both, snap_one = both.save_state(), one.save_state()
    src = rng.randint(-1, B, B)
    both.load_state(snap_both, src=src)
    one.load_state(snap_one, src=src)
    for sim in (both, one):
        sim.observe(aux=True)
    _assert_same(both, one, (preset, team, 'branched'))
    for k in range(4, 9):
        cam, tgt = _actions(cfg, B, k)
        both.step(cam, tgt, aux=True)
        one.step(cam, tgt, aux=True)
        _assert_same(both, one, (preset, team, 'after branching', k))
    both.close()
    one.close()


@pytest.mark.gpu
@pytest.mark.parametrize('fold', ['fast', 'generic'])
@pytest.mark.parametrize('preset', ['MATE-4v8-9.yaml', 'MATE-4v2-0.yaml', 'MATE-8v8-9.yaml'])
def test_every_folded_wrapper_stack(preset, fold, monkeypatch):
    """Every wrapper stack of test_wrappers.py registered with the simulator, on the canonical (fast) and the generic
    shared-memory path: the single team's rows are those of the both-teams environment."""
    import mate_b200
    from test_wrappers import STACKS

    monkeypatch.setenv('MATE_B200_FOLD', '1' if fold == 'fast' else '0')
    monkeypatch.setenv('MATE_B200_REFILL', 'sync')
    B = 300
    for stack in [None] + sorted(STACKS):
        spec = [] if stack is None else STACKS[stack]
        wrappers = [(lambda env, c=cls, k=kw: getattr(mate_b200, c)(env, **k)) for cls, kw in spec]
        for team in ('camera', 'target'):
            for dtype in (torch.float32, torch.float16):
                envs = [mate_b200.make('MultiAgentTracking-v0', config=preset, num_envs=B, max_episode_steps=5, wrappers=wrappers,
                                       observation_dtype=dtype, observed_team=t).unwrapped for t in ('both', team)]
                both, one = (env.sim for env in envs)
                for env in envs:
                    env.reset(seed=8)
                _assert_same(both, one, (preset, stack, team, dtype, 'reset'), snapshot=False)
                for k in range(6):
                    cam, tgt = _actions(both.cfg, B, k)
                    both.step(cam, tgt, auto_reset=True, aux=True)
                    one.step(cam, tgt, auto_reset=True, aux=True)
                    _assert_same(both, one, (preset, stack, team, dtype, k), snapshot=False)
                for env in envs:
                    env.close()


def _lib_call(sim, name, *args):
    with torch.cuda.device(sim.device):
        rc = getattr(sim.lib, name)(sim.handle, *args)
    assert rc == 0, sim.lib.mate_b200_last_error()


@pytest.mark.gpu
@pytest.mark.parametrize('preset', ['MATE-4v8-9.yaml', 'MATE-Navigation.yaml'])
def test_both_pointers_null(preset, monkeypatch):
    """reset, step and observe with no row buffer at all: rewards, done, aux and the state are unchanged."""
    monkeypatch.setenv('MATE_B200_REFILL', 'sync')
    from mate_b200 import _abi
    from mate_b200.sim import _dptr

    B = 777
    cfg, both, none = _sims(preset, B, 'target', max_episode_steps=4)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    both.reset(seed=3)
    none.seed(3)
    _lib_call(none, 'mate_b200_reset', None, none._seed, None, None, stream)   # pylint: disable=protected-access
    none.alloc_aux()
    for k in range(9):
        cam, tgt = _actions(cfg, B, k)
        both.step(cam, tgt, auto_reset=True, aux=True)
        cam_act, tgt_act = none._actions(cam, tgt)   # pylint: disable=protected-access
        _lib_call(none, 'mate_b200_step', _dptr(cam_act), _dptr(tgt_act), None, None, _dptr(none.rewards), _dptr(none.done),
                  ctypes.byref(none._aux_struct), None, _abi.MATE_STEP_AUTO_RESET, stream)   # pylint: disable=protected-access
        torch.cuda.synchronize()
        assert torch.equal(none.rewards, both.rewards) and torch.equal(none.done, both.done), k
        for key, value in both.aux.items():
            assert torch.equal(value, none.aux[key]), (k, key)
    _lib_call(none, 'mate_b200_observe', None, None, ctypes.byref(none._aux_struct), None, stream)   # pylint: disable=protected-access
    both.observe(aux=True)
    torch.cuda.synchronize()
    for key, value in both.aux.items():
        assert torch.equal(value, none.aux[key]), ('observe', key)
    assert _same_snapshots(none, both)
    a, b = both.get_state(), none.get_state()
    for key in a:
        assert np.array_equal(a[key], b[key]), key
    both.close()
    none.close()


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['0', '1', '2'])
@pytest.mark.parametrize('preset', ['MATE-4v8-9.yaml', 'MATE-4v2-9.yaml', 'MATE-Navigation.yaml'])
def test_step_host_single_team(preset, mode, monkeypatch):
    """mate_b200_step_host with one team's buffer NULL on every device -> host leg: the observed buffers hold the rows of
    a both-teams handle, the link carries only the observed team's rows, and a handle that switches a team between NULL
    and a buffer under MATE_STEP_HOST_ROWS_KEPT still fills complete rows."""
    from mate_b200 import _abi
    from mate_b200.config import flatten_config, read_config
    from mate_b200.sim import BatchedSim, _dptr

    monkeypatch.setenv('MATE_B200_HOST_COMPACT', mode)
    monkeypatch.setenv('MATE_B200_REFILL', 'sync')
    cfg = flatten_config(read_config(preset, max_episode_steps=4))
    nc, nt = cfg['num_cameras'], cfg['num_targets']
    B = 2048
    teams = ['target'] + (['camera'] if nc else [])
    ref = BatchedSim(cfg, B, device=0)
    mirror = BatchedSim(cfg, B, device=0)   # both teams, called with the single-team handles' rows_kept pattern
    singles = {team: BatchedSim(cfg, B, device=0, observed_team=team) for team in teams}
    switch = BatchedSim(cfg, B, device=0)   # a both-teams handle whose caller drops and restores a team
    for sim in [ref, mirror, switch] + list(singles.values()):
        sim.reset(seed=9)
    dc, dt = ref.dc, ref.dt

    def buffers():
        return [torch.zeros((B, max(nc, 1), dc)).pin_memory(), torch.zeros((B, nt, dt)).pin_memory(),
                torch.zeros((B, 2)).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory()]

    out_ref, out_mirror, out_switch = buffers(), buffers(), buffers()
    outs = {}
    for team in teams:
        out = buffers()
        out[0 if team == 'target' else 1] = None
        outs[team] = out
    row_bytes = {'camera': B * nc * dc * 4, 'target': B * nt * dt * 4}
    rng = np.random.RandomState(3)
    for k in range(12):
        cam_act = torch.from_numpy((rng.uniform(-1, 1, (B, max(nc, 1), 2)) * [5.0, 2.5]).astype(np.float32)).pin_memory()
        tgt_act = torch.from_numpy((rng.uniform(-1, 1, (B, nt, 2)) * 20.0).astype(np.float32)).pin_memory()
        ref.step_host(cam_act, tgt_act, out_ref, rows_kept=False)
        mirror.step_host(cam_act, tgt_act, out_mirror, rows_kept=(k % 4 != 0))
        leg_mirror, link_mirror = mirror.host_leg_info()
        links = 0
        for team in teams:
            singles[team].step_host(cam_act, tgt_act, outs[team], rows_kept=(k % 4 != 0))
            leg, link = singles[team].host_leg_info()
            slot = 0 if team == 'camera' else 1
            assert torch.equal(outs[team][slot], out_ref[slot]), (team, k)
            assert torch.equal(outs[team][2], out_ref[2]) and torch.equal(outs[team][3], out_ref[3]), (team, k)
            assert leg == leg_mirror, (team, k)
            if leg == 0:
                assert link == row_bytes[team], (team, k)
            links += link
        # each team's rows are compacted on their own: the single-team links add up to the both-teams link
        assert links == link_mirror, (k, links, link_mirror)
        # the switching caller: every third call drops a team (its buffer keeps what it held), the next call restores
        # it with rows_kept=True -- the library must notice the pointer change and write the complete rows
        dropped = (k % 3 == 1)
        drop = 1 if (k // 3) % 2 == 0 or not nc else 0
        call = list(out_switch)
        if dropped:
            call[drop] = None
            out_switch[drop].fill_(-9.0)   # stale content the next call must overwrite
        # the C call takes NULL for any team; BatchedSim.step_host refuses None for a team its handle observes
        with torch.cuda.device(switch.device):
            rc = switch.lib.mate_b200_step_host(switch.handle, _dptr(cam_act) if nc else None, _dptr(tgt_act), _dptr(call[0]) if nc else None,
                                                _dptr(call[1]), _dptr(call[2]), _dptr(call[3]), _abi.MATE_STEP_HOST_ROWS_KEPT | _abi.MATE_STEP_AUTO_RESET)
        assert rc == 0, switch.lib.mate_b200_last_error()
        for slot in range(2):
            if (slot == 0 and not nc) or (dropped and slot == drop):
                continue
            assert torch.equal(out_switch[slot], out_ref[slot]), ('switch', slot, k)
        leg, link = switch.host_leg_info()
        if dropped and leg == 0:
            assert link == row_bytes['target' if drop == 0 else 'camera'], ('switch link', k)
    for sim in [ref, mirror, switch] + list(singles.values()):
        sim.close()


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', [torch.float32, torch.float16])
def test_device_memory_drops_by_the_unobserved_rows(dtype):
    from mate_b200.config import flatten_config, read_config
    from mate_b200.sim import BatchedSim

    cfg = flatten_config(read_config('MATE-4v8-9.yaml'))
    B = 4096
    size = 2 if dtype == torch.float16 else 4
    used = {}
    for team in ('both', 'camera', 'target'):
        gc.collect()   # nothing left over from earlier tests is freed while a handle is created
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        sim = BatchedSim(cfg, B, device=0, observation_dtype=dtype, observed_team=team)
        used[team] = torch.cuda.memory_allocated() - before
        if team == 'both':
            rows = {'camera': sim.cam_obs.numel() * size, 'target': sim.tgt_obs.numel() * size}
        sim.close()
        del sim
    assert rows['camera'] == B * 4 * 126 * size and rows['target'] == B * 8 * 131 * size
    assert used['both'] - used['camera'] == rows['target']
    assert used['both'] - used['target'] == rows['camera']


def _camera_stack(observed_team, B):
    import mate_b200 as mate

    return mate.make('MATE-4v8-9-v0', num_envs=B, observed_team=observed_team, wrappers=[
        mate.MoreTrainingInformation, mate.RepeatedRewardIndividualDone,
        lambda e: mate.AuxiliaryCameraRewards(e, coefficients={'raw_reward': 1.0, 'coverage_rate': 1.0}, reduction='mean'),
        lambda e: mate.MultiCamera(e, target_agent=mate.GreedyTargetAgent(seed=0))])


def _assert_infos_equal(a, b, ctx):
    assert set(a) == set(b), (ctx, set(a) ^ set(b))
    for key, value in a.items():
        if torch.is_tensor(value):
            assert torch.equal(value, b[key]), (ctx, key)
        else:
            assert np.array_equal(np.asarray(value), np.asarray(b[key])), (ctx, key)


@pytest.mark.gpu
def test_multi_camera_stack_for_200_steps():
    """The README's MultiCamera stack: camera observations, rewards and infos equal those of the both-teams stack, the
    opponent observation is None, and MoreTrainingInformation leaves out only 'target_states'."""
    B = 512
    env_both, env_cam = _camera_stack('both', B), _camera_stack('camera', B)
    obs_both, obs_cam = env_both.reset(seed=3), env_cam.reset(seed=3)
    assert torch.equal(obs_both, obs_cam)
    assert env_cam.opponent_joint_observation is None and env_both.opponent_joint_observation is not None
    rng = np.random.RandomState(5)
    for k in range(200):
        act = torch.from_numpy((rng.uniform(-1, 1, (B, 4, 2)) * [5.0, 2.5]).astype(np.float32)).cuda()
        obs_both, rew_both, done_both, infos_both = env_both.step(act)
        obs_cam, rew_cam, done_cam, infos_cam = env_cam.step(act)
        assert torch.equal(obs_both, obs_cam) and torch.equal(rew_both, rew_cam) and torch.equal(done_both, done_cam), k
        assert 'target_states' in infos_both and 'target_states' not in infos_cam and 'camera_states' in infos_cam, k
        infos_both = dict(infos_both)
        del infos_both['target_states']
        _assert_infos_equal(infos_both, infos_cam, k)
        assert env_cam.opponent_joint_observation is None
    env_both.unwrapped.close()
    env_cam.unwrapped.close()


@pytest.mark.gpu
def test_more_training_information_under_target_observation():
    import mate_b200 as mate

    B = 128
    envs = [mate.make('MATE-4v8-9-v0', num_envs=B, observed_team=t, wrappers=[mate.MoreTrainingInformation]) for t in ('both', 'target')]
    for env in envs:
        env.reset(seed=1)
    cam = torch.zeros((B, 4, 2), device='cuda')
    tgt = torch.ones((B, 8, 2), device='cuda')
    (c0, t0), _, _, (ci0, ti0) = envs[0].step((cam, tgt))
    (c1, t1), _, _, (ci1, ti1) = envs[1].step((cam, tgt))
    assert c1 is None and torch.equal(t0, t1)
    assert 'camera_states' not in ci1 and 'camera_states' not in ti1 and torch.equal(ti0['target_states'], ti1['target_states'])
    assert set(ci0) - set(ci1) == {'camera_states'}
    with pytest.raises(ValueError, match='camera rows'):
        mate.MultiTarget(envs[1], camera_agent=mate.GreedyCameraAgent(seed=0))
    from mate_b200 import _abi

    sim = envs[1].unwrapped.sim
    sim.set_observation_wrappers([_abi.OBS_RESCALED])
    with pytest.raises(ValueError, match="both teams' rows"):   # the separate wrapper pass needs both teams' rows
        sim.transform_observations()
    from mate_b200.sim import _dptr

    both_sim = envs[0].unwrapped.sim   # and the C call still refuses a NULL row pointer (MATE_EINVAL)
    rows = torch.zeros_like(both_sim.cam_obs)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    aff = torch.zeros((both_sim.dt, 2), device='cuda')
    assert both_sim.lib.mate_b200_transform_observations(both_sim.handle, None, _dptr(both_sim.tgt_obs), sim._obs_ops_c, 1,  # pylint: disable=protected-access
                                                         None, _dptr(aff), stream) == -1
    assert both_sim.lib.mate_b200_transform_observations(both_sim.handle, _dptr(rows), None, sim._obs_ops_c, 1,  # pylint: disable=protected-access
                                                         _dptr(aff), _dptr(aff), stream) == -1
    for env in envs:
        env.unwrapped.close()


@pytest.mark.gpu
def test_snapshot_resume_under_camera_observation(tmp_path):
    """A camera-observing MultiCamera stack saved, torch.save'd, loaded into a fresh stack and resumed continues bit for
    bit like the stack that was never interrupted."""
    B = 256
    env, resumed = _camera_stack('camera', B), _camera_stack('camera', B)
    env.reset(seed=4)
    resumed.reset(seed=99)
    rng = np.random.RandomState(6)
    acts = [torch.from_numpy((rng.uniform(-1, 1, (B, 4, 2)) * [5.0, 2.5]).astype(np.float32)).cuda() for _ in range(40)]
    for act in acts[:15]:
        env.step(act)
    path = tmp_path / 'snap.pt'
    torch.save(env.save_state(), path)
    obs = resumed.load_state(torch.load(path), resume=True)
    assert torch.equal(obs, env.unwrapped.sim.cam_obs) and resumed.opponent_joint_observation is None
    for k, act in enumerate(acts[15:]):
        a = env.step(act)
        b = resumed.step(act)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]), k
    env.unwrapped.close()
    resumed.unwrapped.close()
