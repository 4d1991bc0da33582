"""float16 observation rows (mate_b200_set_observation_format): on every path that writes rows they are, bit for bit,
the float32 rows of the same call rounded once to nearest even (``rows.to(torch.float16)``); everything else a call
returns is the same as for float32 rows."""

import os
import re

import numpy as np
import pytest

torch = pytest.importorskip('torch')

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRESETS = [f'MATE-{nc}v{nt}-{no}.yaml' for nc, nt in ((1, 1), (1, 2), (2, 2), (2, 4), (4, 2), (4, 4), (4, 8), (8, 8))
           for no in (0, 9)] + ['MATE-Navigation.yaml']


# ---------------------------------------------------------------------------------------------- CPU
def test_header_format_codes_match_the_binding():
    from mate_b200 import _abi

    text = open(os.path.join(ROOT, 'include', 'mate_b200.h'), encoding='UTF-8').read()
    codes = dict(re.findall(r'#define (MATE_OBS_FORMAT_F\d+) (\d+)', text))
    assert codes == {'MATE_OBS_FORMAT_F32': str(_abi.MATE_OBS_FORMAT_F32), 'MATE_OBS_FORMAT_F16': str(_abi.MATE_OBS_FORMAT_F16)}


def test_observation_dtype_is_checked_before_anything_is_allocated():
    from mate_b200.config import flatten_config, read_config
    from mate_b200.environment import MultiAgentTracking
    from mate_b200.sim import BatchedSim

    cfg = flatten_config(read_config('MATE-4v8-9.yaml'))
    for dtype in (torch.bfloat16, torch.float64, 'float16'):
        with pytest.raises(ValueError):
            BatchedSim(cfg, 16, observation_dtype=dtype)
        with pytest.raises(ValueError):
            MultiAgentTracking('MATE-4v8-9.yaml', num_envs=16, observation_dtype=dtype)
    with pytest.raises(ValueError):   # the single-environment mode returns the reference's float64 NumPy rows
        MultiAgentTracking('MATE-4v8-9.yaml', observation_dtype=torch.float16)


# ---------------------------------------------------------------------------------------------- GPU
def _bits_equal(rows32, rows16):
    """rows16 holds exactly rows32 rounded to float16 (compared as bit patterns: -0.0 and 0.0 differ)."""
    assert rows16.dtype == torch.float16 and rows32.dtype == torch.float32
    return torch.equal(rows32.to(torch.float16).view(torch.int16), rows16.view(torch.int16))


def _pair(preset, B, **overrides):
    from mate_b200.config import flatten_config, read_config
    from mate_b200.sim import BatchedSim

    cfg = flatten_config(read_config(preset, **overrides))
    return cfg, BatchedSim(cfg, B, device=0), BatchedSim(cfg, B, device=0, observation_dtype=torch.float16)


def _actions(cfg, B, k):
    gen = torch.Generator(device='cuda')
    gen.manual_seed(1000 + k)
    scale = torch.tensor([cfg['camera_rotation_step'], cfg['camera_zooming_step']], device='cuda')
    cam = (torch.rand((B, max(cfg['num_cameras'], 1), 2), device='cuda', generator=gen) * 2 - 1) * scale
    tgt = (torch.rand((B, cfg['num_targets'], 2), device='cuda', generator=gen) * 2 - 1) * cfg['target_step_size']
    return cam[:, :cfg['num_cameras']].contiguous(), tgt


def _assert_same_call(a, b, ctx, aux=True):
    torch.cuda.synchronize()
    assert _bits_equal(a.cam_obs, b.cam_obs), (ctx, 'cam_obs')
    assert _bits_equal(a.tgt_obs, b.tgt_obs), (ctx, 'tgt_obs')
    assert torch.equal(a.rewards, b.rewards) and torch.equal(a.done, b.done), ctx
    if aux:
        for key, value in a.aux.items():
            assert torch.equal(value, b.aux[key]), (ctx, key)


def _run_steps(cfg, a, b, B, steps, tag):
    for k in range(steps):
        cam, tgt = _actions(cfg, B, k)
        a.step(cam, tgt, auto_reset=True, aux=True)
        b.step(cam, tgt, auto_reset=True, aux=True)
        _assert_same_call(a, b, (tag, k))


@pytest.mark.gpu
@pytest.mark.parametrize('refill', ['sync', 'default'])
@pytest.mark.parametrize('preset', PRESETS)
def test_every_preset_writes_the_rounded_float32_rows(preset, refill, monkeypatch):
    """A ragged batch (not a multiple of the warp tile) with episodes short enough that most environments auto-reset,
    from the prepared next episodes (refilled after every step, or on the side stream)."""
    if refill == 'sync':
        monkeypatch.setenv('MATE_B200_REFILL', 'sync')
    else:
        monkeypatch.delenv('MATE_B200_REFILL', raising=False)
    B = 1001
    cfg, a, b = _pair(preset, B, max_episode_steps=4)
    a.reset(seed=11)
    b.reset(seed=11)
    _assert_same_call(a, b, (preset, 'reset'), aux=False)
    _run_steps(cfg, a, b, B, 11, preset)
    assert int(a.episode_stats()[0]) >= B    # the auto-reset paths ran
    a.close()
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize('tile', ['32', '16', '8'])
def test_full_size_4v8_9(tile, monkeypatch):
    """MATE-4v8-9 x 65 536 with the asynchronous refill and every warp tile size."""
    monkeypatch.setenv('MATE_B200_TILE', tile)
    monkeypatch.delenv('MATE_B200_REFILL', raising=False)
    B = 65536
    cfg, a, b = _pair('MATE-4v8-9.yaml', B, max_episode_steps=5)
    a.reset(seed=2)
    b.reset(seed=2)
    _assert_same_call(a, b, ('full', 'reset'), aux=False)
    _run_steps(cfg, a, b, B, 8, ('full', tile))
    a.close()
    b.close()


@pytest.mark.gpu
@pytest.mark.parametrize('fold', ['fast', 'generic'])
@pytest.mark.parametrize('preset', ['MATE-4v8-9.yaml', 'MATE-4v2-0.yaml', 'MATE-8v8-9.yaml'])
def test_masked_reset_observe_and_registered_wrappers(preset, fold, monkeypatch):
    """reset(env_mask), observe() after set_state, and every wrapper stack of test_wrappers.py registered on both
    simulators (applied by the packer before the rows are rounded)."""
    import mate_b200
    from test_wrappers import STACKS

    monkeypatch.setenv('MATE_B200_FOLD', '1' if fold == 'fast' else '0')
    monkeypatch.setenv('MATE_B200_REFILL', 'sync')
    B = 300
    rng = np.random.RandomState(4)
    for stack in [None] + sorted(STACKS):
        spec = [] if stack is None else STACKS[stack]
        wrappers = [(lambda env, c=cls, k=kw: getattr(mate_b200, c)(env, **k)) for cls, kw in spec]
        envs = [mate_b200.make('MultiAgentTracking-v0', config=preset, num_envs=B, max_episode_steps=5, wrappers=wrappers,
                               observation_dtype=dtype).unwrapped for dtype in (torch.float32, torch.float16)]
        a, b = (env.sim for env in envs)
        assert b.cam_obs.dtype == torch.float16 and envs[1].observation_dtype == torch.float16
        for env in envs:
            env.reset(seed=8)
        _assert_same_call(a, b, (preset, stack, 'reset'))
        _run_steps(a.cfg, a, b, B, 6, (preset, stack))
        mask = torch.from_numpy(rng.randint(0, 2, B).astype(np.uint8)).cuda()
        a.reset(env_mask=mask)
        b.reset(env_mask=mask)
        _assert_same_call(a, b, (preset, stack, 'masked reset'), aux=False)
        state = a.get_state()
        for sim in (a, b):
            sim.set_state(state)
            sim.observe(aux=True)
        _assert_same_call(a, b, (preset, stack, 'observe after set_state'))
        for env in envs:
            env.close()


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['0', '1', '2'])
@pytest.mark.parametrize('preset', ['MATE-4v8-9.yaml', 'MATE-4v2-9.yaml', 'MATE-8v8-9.yaml', 'MATE-Navigation.yaml'])
def test_step_host_float16_rows(preset, mode, monkeypatch):
    """mate_b200_step_host into float16 pinned buffers, on every device -> host leg, with and without
    MATE_STEP_HOST_ROWS_KEPT, including a caller that scribbles over its buffers and one that swaps them: the buffers
    hold the device float16 step's rows byte for byte.  The dense leg moves exactly half the bytes of float32 rows."""
    from mate_b200.config import flatten_config, read_config
    from mate_b200.sim import BatchedSim

    monkeypatch.setenv('MATE_B200_HOST_COMPACT', mode)
    monkeypatch.setenv('MATE_B200_REFILL', 'sync')
    cfg = flatten_config(read_config(preset, max_episode_steps=4))
    nc, nt = cfg['num_cameras'], cfg['num_targets']
    B = 2048
    dev16, host16 = (BatchedSim(cfg, B, device=0, observation_dtype=torch.float16) for _ in range(2))
    host32 = BatchedSim(cfg, B, device=0)
    for sim in (dev16, host16, host32):
        sim.reset(seed=9)

    def buffers(dtype):
        return (torch.zeros((B, max(nc, 1), dev16.dc), dtype=dtype).pin_memory(), torch.zeros((B, nt, dev16.dt), dtype=dtype).pin_memory(),
                torch.zeros((B, 2)).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory())

    out, other, out32 = buffers(torch.float16), buffers(torch.float16), buffers(torch.float32)
    rng = np.random.RandomState(3)
    legs = set()
    for k in range(14):
        cam_act = torch.from_numpy((rng.uniform(-1, 1, (B, max(nc, 1), 2)) * [5.0, 2.5]).astype(np.float32)).pin_memory()
        tgt_act = torch.from_numpy((rng.uniform(-1, 1, (B, nt, 2)) * 20.0).astype(np.float32)).pin_memory()
        (cam, tgt), rew, done = dev16.step(cam_act.cuda(), tgt_act.cuda(), auto_reset=True)
        if k == 6:     # the caller scribbles over the buffers and says so by not passing the flag
            out[0].fill_(7.0)
            out[1].fill_(-3.0)
            host16.step_host(cam_act, tgt_act, out, auto_reset=True, rows_kept=False)
        elif k == 10:  # other buffers: the flag is passed wrongly, the library notices the new addresses
            other[0].fill_(5.0)
            other[1].fill_(5.0)
            out, other = other, out
            host16.step_host(cam_act, tgt_act, out, auto_reset=True, rows_kept=True)
        else:
            host16.step_host(cam_act, tgt_act, out, auto_reset=True, rows_kept=(k != 3))
        leg16, link16 = host16.host_leg_info()
        host32.step_host(cam_act, tgt_act, out32, auto_reset=True, rows_kept=False)
        leg32, link32 = host32.host_leg_info()
        torch.cuda.synchronize()
        legs.add(leg16)
        if nc:
            assert torch.equal(cam.cpu().view(torch.int16), out[0].view(torch.int16)), k
            assert _bits_equal(out32[0], out[0]), k
        assert torch.equal(tgt.cpu().view(torch.int16), out[1].view(torch.int16)), k
        assert _bits_equal(out32[1], out[1]), k
        assert torch.equal(rew.cpu(), out[2]) and torch.equal(done.cpu(), out[3]), k
        assert torch.equal(out32[2], out[2]) and torch.equal(out32[3], out[3]), k
        if leg16 == 0 and leg32 == 0:
            assert 2 * link16 == link32 == B * (nc * dev16.dc + nt * dev16.dt) * 4, k
    if mode == '0':
        assert legs == {0}
    for sim in (dev16, host16, host32):
        sim.close()


@pytest.mark.gpu
def test_make_with_single_team_wrappers_and_load_config():
    """mate.make(..., observation_dtype=torch.float16) with RescaledObservation and MultiTarget(GreedyCameraAgent):
    the greedy cameras read the target flags of the float16 camera rows and act exactly as on float32 rows, so rewards
    and done agree for 200 steps.  load_config keeps the dtype."""
    import mate_b200

    B = 256

    def make(dtype):
        return mate_b200.make('MATE-4v8-9-v0', num_envs=B, observation_dtype=dtype, wrappers=[
            mate_b200.RescaledObservation, lambda e: mate_b200.MultiTarget(e, camera_agent=mate_b200.GreedyCameraAgent(seed=1))])

    env32, env16 = make(torch.float32), make(torch.float16)
    obs32, obs16 = env32.reset(seed=6), env16.reset(seed=6)
    assert obs16.dtype == torch.float16 and _bits_equal(obs32, obs16)
    rng = np.random.RandomState(2)
    for k in range(200):
        act = torch.from_numpy((rng.uniform(-1, 1, (B, 8, 2)) * 20.0).astype(np.float32)).cuda()
        obs32, rew32, done32, _ = env32.step(act)
        obs16, rew16, done16, _ = env16.step(act)
        assert torch.equal(rew32, rew16) and torch.equal(done32, done16), k
        assert _bits_equal(obs32, obs16), k
        assert torch.equal(env32.opponent_agent.actions, env16.opponent_agent.actions), k
    base = env16.unwrapped
    base.load_config()
    assert base.observation_dtype == torch.float16 and base.sim.tgt_obs.dtype == torch.float16
    env32.unwrapped.close()
    base.close()


@pytest.mark.gpu
def test_errors():
    from mate_b200 import _abi

    cfg, a, b = _pair('MATE-4v8-9.yaml', 64)
    lib = b.lib
    assert lib.mate_b200_set_observation_format(b.handle, 7) == -1                          # unknown code: MATE_EINVAL
    assert lib.mate_b200_set_observation_format(b.handle, _abi.MATE_OBS_FORMAT_F16) == 0    # before the first reset: allowed
    b.set_observation_wrappers([_abi.OBS_RESCALED])
    b.reset(seed=1)
    with pytest.raises(ValueError):   # the separate float32 pass refuses float16 rows
        b.transform_observations()
    rc = lib.mate_b200_set_observation_format(b.handle, _abi.MATE_OBS_FORMAT_F32)
    assert rc == -4 and b'before' in lib.mate_b200_last_error()                            # MATE_ESTATE after a reset
    assert b.cam_obs.dtype == torch.float16
    out32 = (torch.zeros((64, 4, b.dc)).pin_memory(), torch.zeros((64, 8, b.dt)).pin_memory(),
             torch.zeros((64, 2)).pin_memory(), torch.zeros(64, dtype=torch.uint8).pin_memory())
    cam, tgt = _actions(cfg, 64, 0)
    with pytest.raises(ValueError):
        b.step_host(cam.cpu(), tgt.cpu(), out32)
    a.step_host(cam.cpu(), tgt.cpu(), out32)   # the same buffers are right for a float32 simulator
    a.close()
    b.close()
