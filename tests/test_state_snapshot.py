"""Device-side state snapshots (mate_b200_save_state / mate_b200_load_state): a whole-batch save followed by a resume
continues bit for bit, on the same handle and on a fresh one; a load through an index map branches environments from
others and leaves the unmapped ones untouched; the single-team wrappers carry their opponents' state along."""

import gc
import io
import os
import re

import numpy as np
import pytest

torch = pytest.importorskip('torch')

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRESETS = [f'MATE-{nc}v{nt}-{no}.yaml' for nc, nt in ((1, 1), (1, 2), (2, 2), (2, 4), (4, 2), (4, 4), (4, 8), (8, 8))
           for no in (0, 9)] + ['MATE-Navigation.yaml']


def _header(**fields):
    from mate_b200 import _abi

    values = dict(version=_abi.MATE_SNAPSHOT_VERSION, num_cameras=4, num_targets=8, num_obstacles=9, count=4,
                  config_hash=0x0123456789ABCDEF, seed=(1 << 64) - 3, payload_bytes=4096)
    values.update(fields)
    return values


# ---------------------------------------------------------------------------------------------- CPU
def test_header_snapshot_codes_match_the_binding():
    from mate_b200 import _abi

    text = open(os.path.join(ROOT, 'include', 'mate_b200.h'), encoding='UTF-8').read()
    codes = dict(re.findall(r'#define (MATE_SNAPSHOT_VERSION|MATE_LOAD_STATE_RESUME) (\d+)u?', text))
    assert codes == {'MATE_SNAPSHOT_VERSION': str(_abi.MATE_SNAPSHOT_VERSION), 'MATE_LOAD_STATE_RESUME': str(_abi.MATE_LOAD_STATE_RESUME)}
    import ctypes

    assert ctypes.sizeof(_abi.MateSnapshotInfo) == 6 * 4 + 3 * 8


def test_snapshot_survives_torch_save_and_load():
    from mate_b200.sim import StateSnapshot

    payload = torch.arange(4096, dtype=torch.int64).to(torch.uint8)
    snap = StateSnapshot(payload, py_seed=77, extras={'environment': {'seed': 5, 'np_random': ('MT19937', torch.arange(624), 3, 0, 0.0)}},
                         **_header())
    buf = io.BytesIO()
    torch.save(snap, buf)
    buf.seek(0)
    back = torch.load(buf)   # weights_only, the default
    assert isinstance(back, StateSnapshot)
    assert torch.equal(back.payload, payload) and back.payload.dtype == torch.uint8
    for name, value in _header().items():
        assert getattr(back, name) == value, name
    assert back.py_seed == 77
    assert back.extras['environment']['seed'] == 5 and torch.equal(back.extras['environment']['np_random'][1], torch.arange(624))
    info = back.info()
    assert info.seed == (1 << 64) - 3 and info.config_hash == 0x0123456789ABCDEF and info.count == 4


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f'{name} was called: host indices must be checked before any library call')


def test_host_index_lists_are_checked_before_any_library_call():
    from mate_b200.sim import BatchedSim, StateSnapshot

    sim = BatchedSim.__new__(BatchedSim)   # no device: every check below has to happen on the host
    sim.B, sim.device, sim.lib, sim.handle, sim._seed = 8, torch.device('cuda', 0), _NoLibrary(), None, 0
    for envs in ([0, 8], [-1, 2], [0.0, 1.0], [], [[0, 1]], np.array([True, False]), torch.tensor([1.5])):
        with pytest.raises(ValueError):
            sim.save_state(envs)
    snap = StateSnapshot(torch.zeros(16, dtype=torch.uint8), **_header(count=4))
    for src in ([0] * 7, [0] * 9, [0, 1, 2, 3, 4, 0, 0, 0], [0.0] * 8, np.zeros((2, 4), dtype=np.int64), torch.zeros(8)):
        with pytest.raises(ValueError):
            sim.load_state(snap, src=src)


# ---------------------------------------------------------------------------------------------- GPU
def _cfg(preset, **overrides):
    from mate_b200.config import flatten_config, read_config

    return flatten_config(read_config(preset, **overrides))


def _actions(cfg, B, k):
    """Seeded random joint actions of step k (device tensors)."""
    gen = torch.Generator(device='cuda')
    gen.manual_seed(1000 + k)
    nc, nt = cfg['num_cameras'], cfg['num_targets']
    cam = None
    if nc:
        scale = torch.tensor([cfg['camera_rotation_step'], cfg['camera_zooming_step']], device='cuda')
        cam = (torch.rand((B, nc, 2), generator=gen, device='cuda') * 2 - 1) * scale
    tgt = (torch.rand((B, nt, 2), generator=gen, device='cuda') * 2 - 1) * cfg['target_step_size']
    return cam, tgt


def _step(sim, cfg, k):
    cam, tgt = _actions(cfg, sim.B, k)
    sim.step(cam, tgt, auto_reset=True, aux=True)


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.float16 else t


def _assert_same_step(a, b):
    """Observation rows (b's in b's format), rewards, done and every MateStepAux field of the last step, bitwise."""
    for rows_a, rows_b in ((a.cam_obs, b.cam_obs), (a.tgt_obs, b.tgt_obs)):
        assert torch.equal(_bits(rows_a.to(rows_b.dtype)), _bits(rows_b))
    assert torch.equal(a.rewards.view(torch.int32), b.rewards.view(torch.int32))
    assert torch.equal(a.done, b.done)
    for name, value in a.aux.items():
        other = b.aux[name]
        assert torch.equal(value.view(torch.uint8) if value.dtype == torch.float32 else value,
                           other.view(torch.uint8) if other.dtype == torch.float32 else other), name


def _assert_same_stats(a, b, all_entries):
    sa, sb = a.episode_stats().cpu().numpy(), b.episode_stats().cpu().numpy()
    np.testing.assert_array_equal(sa[[0, 1, 2, 3, 5]], sb[[0, 1, 2, 3, 5]])
    # Entry 4 adds one non-integer float32 (an episode's mean coverage) per finished episode with atomics whose order is
    # not fixed, so two identical runs differ in rounding: each add rounds by at most half an ulp of the running sum, in
    # each run.  (Measured on a B200: up to 5.7e-6 relative for MATE-4v8-9 x 65 536.)
    bound = sa[0] * np.finfo(np.float32).eps * max(abs(sa[4]), abs(sb[4]))
    assert abs(float(sa[4]) - float(sb[4])) <= bound, (sa[4], sb[4], bound)
    if all_entries:   # prepared / in-place auto-resets: the same only when the refill runs after every step
        np.testing.assert_array_equal(sa[6:8], sb[6:8])


@pytest.mark.gpu
@pytest.mark.parametrize('preset', PRESETS)
def test_save_load_round_trip_every_preset(preset):
    """Save after 30 steps (with auto-resets), step 40 more, resume: saving again gives the same bytes and get_state the
    same arrays as at save time."""
    from mate_b200.sim import BatchedSim

    cfg = _cfg(preset, max_episode_steps=12)
    B = 1000
    sim = BatchedSim(cfg, B, device=0)
    sim.reset(seed=3)
    for k in range(30):
        _step(sim, cfg, k)
    snap = sim.save_state()
    assert snap.count == B and snap.payload.numel() == snap.payload_bytes == sim.snapshot_bytes(B)
    view = sim.get_state()
    first = snap.payload.clone()
    for k in range(30, 70):
        _step(sim, cfg, k)
    sim.load_state(snap, resume=True)   # the statistics at the end of the payload come back too
    assert torch.equal(sim.save_state().payload, first)
    for name, value in sim.get_state().items():
        np.testing.assert_array_equal(value, view[name], err_msg=name)
    sim.close()


RESUME_CASES = [('MATE-4v8-9.yaml', 65536, mode, torch.float32, torch.float32) for mode in ('sync', 'default', 'off')]
RESUME_CASES += [(preset, 4096, mode, torch.float32, torch.float32) for preset in
                 ('MATE-8v8-9.yaml', 'MATE-4v8-0.yaml', 'MATE-4v2-9.yaml', 'MATE-Navigation.yaml') for mode in ('sync', 'default', 'off')]
RESUME_CASES += [('MATE-4v8-9.yaml', 4096, 'sync', torch.float32, torch.float16), ('MATE-4v8-9.yaml', 4096, 'default', torch.float16, torch.float16)]


@pytest.mark.gpu
@pytest.mark.parametrize('preset,B,refill,saving_dtype,loading_dtype', RESUME_CASES)
def test_resume_replays_bit_for_bit(monkeypatch, preset, B, refill, saving_dtype, loading_dtype):
    """A resume snapshot taken at step k, loaded into a fresh handle (same configuration, batch and env_index_base) and
    into the saving handle itself, replays steps k..N of the original run exactly."""
    from mate_b200.sim import BatchedSim

    if refill != 'default':
        monkeypatch.setenv('MATE_B200_REFILL', refill)
    cfg = _cfg(preset, max_episode_steps=9)
    k0, n = 10, 30
    a = BatchedSim(cfg, B, device=0, observation_dtype=saving_dtype)
    b = BatchedSim(cfg, B, device=0, observation_dtype=loading_dtype)
    a.reset(seed=11)
    for k in range(k0):
        _step(a, cfg, k)
    snap = a.save_state()
    # (b) a fresh handle, in lockstep with the original run
    b.load_state(snap, resume=True)
    for k in range(k0, n):
        _step(a, cfg, k)
        _step(b, cfg, k)
        _assert_same_step(a, b)
    _assert_same_stats(a, b, refill == 'sync')
    # (a) the saving handle, in lockstep with the original run made again from the start
    a.load_state(snap, resume=True)
    c = b if loading_dtype == saving_dtype else BatchedSim(cfg, B, device=0, observation_dtype=saving_dtype)
    c.episode_stats(reset_after=True)
    c.reset(seed=11)
    for k in range(k0):
        _step(c, cfg, k)
    for k in range(k0, n):
        _step(a, cfg, k)
        _step(c, cfg, k)
        _assert_same_step(c, a)
    _assert_same_stats(a, c, refill == 'sync')
    for sim in {id(s): s for s in (a, b, c)}.values():
        sim.close()


def _branch_map(B, seed):
    """A random map with repeats and -1 entries whose sources keep their own state (src[s] == s for every source s)."""
    rng = np.random.default_rng(seed)
    sources = rng.choice(B, 64, replace=False)
    src = np.where(rng.random(B) < 0.2, -1, rng.choice(sources, B))
    src[sources] = sources
    return src


@pytest.mark.gpu
def test_branching_load_copies_mapped_environments_and_keeps_the_others():
    from mate_b200.sim import BatchedSim

    cfg = _cfg('MATE-4v8-9.yaml')
    B = 4096
    sim = BatchedSim(cfg, B, device=0)
    sim.reset(seed=2)
    for k in range(20):
        _step(sim, cfg, k)
    src = _branch_map(B, 5)
    mapped, kept = np.nonzero(src >= 0)[0], np.nonzero(src < 0)[0]
    snap = sim.save_state()
    view = sim.get_state()
    sources_before = sim.save_state(src[mapped]).payload.clone()
    kept_before = sim.save_state(kept).payload.clone()
    sim.load_state(snap, src=torch.from_numpy(src).cuda())   # device map: no host check, no synchronisation
    after = sim.get_state()
    for name, value in after.items():
        np.testing.assert_array_equal(value[mapped], view[name][src[mapped]], err_msg=name)
        np.testing.assert_array_equal(value[kept], view[name][kept], err_msg=name)
    assert torch.equal(sim.save_state(mapped).payload, sources_before)   # every state array, bit for bit
    assert torch.equal(sim.save_state(kept).payload, kept_before)
    # one step later, with the same actions and draws for a clone and its source, the clone's outputs are its source's
    origin = torch.from_numpy(np.where(src >= 0, src, np.arange(B))).cuda()
    cam, tgt = _actions(cfg, B, 99)
    replay = (np.ones((B, 4, 8), dtype=np.uint8), np.zeros((B, 8), dtype=np.int8))
    sim.step(cam[origin], tgt[origin], auto_reset=True, replay=replay)
    idx = torch.from_numpy(mapped).cuda()
    for value in (sim.cam_obs, sim.tgt_obs, sim.rewards, sim.done):
        assert torch.equal(value[idx], value[origin[idx]])
    sim.close()


@pytest.mark.gpu
@pytest.mark.parametrize('compact', ['0', '1', '2'])
def test_load_between_step_host_calls(monkeypatch, compact):
    """A branching load between two step_host calls: the next calls (rows kept on the device, changes only) give the
    rows step gives on a twin handle loaded the same way."""
    from mate_b200.sim import BatchedSim

    monkeypatch.setenv('MATE_B200_HOST_COMPACT', compact)
    cfg = _cfg('MATE-4v8-9.yaml', max_episode_steps=15)
    B = 4096
    host, twin = BatchedSim(cfg, B, device=0), BatchedSim(cfg, B, device=0)
    out = (torch.zeros((B, 4, host.dc)).pin_memory(), torch.zeros((B, 8, host.dt)).pin_memory(),
           torch.zeros((B, 2)).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory())
    for sim in (host, twin):
        sim.reset(seed=4)

    def both(k, rows_kept):
        cam, tgt = _actions(cfg, B, k)
        host.step_host(cam.cpu().pin_memory(), tgt.cpu().pin_memory(), out, auto_reset=True, rows_kept=rows_kept)
        twin.step(cam, tgt, auto_reset=True)
        for got, want in zip(out, (twin.cam_obs, twin.tgt_obs, twin.rewards, twin.done)):
            assert torch.equal(got, want.cpu())

    for k in range(8):
        both(k, rows_kept=k > 0)
    snap = host.save_state()
    torch.cuda.synchronize()
    src = torch.from_numpy(_branch_map(B, 8))
    host.load_state(snap, src=src)
    twin.load_state(snap, src=src)
    for k in range(8, 14):
        both(k, rows_kept=True)
    if compact != '0':
        assert host.host_leg_info()[0] == 2
    host.close()
    twin.close()


def _wrapped(kind):
    import mate_b200

    env = mate_b200.make('MultiAgentTracking-v0', config='MATE-4v8-9.yaml', num_envs=4096, max_episode_steps=25)
    if kind == 'camera':
        return mate_b200.MultiCamera(env, target_agent=mate_b200.GreedyTargetAgent(seed=3))
    return mate_b200.MultiTarget(env, camera_agent=mate_b200.GreedyCameraAgent(seed=3))


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['camera', 'target'])
def test_single_team_wrappers_resume_and_branch(kind):
    env = _wrapped(kind)
    base = env.unwrapped
    cfg = base.flat_config
    B, team = base.num_envs, (0 if kind == 'camera' else 1)
    agent = env.opponent_agent
    env.reset(seed=6)

    def run(first, last):
        out = []
        for k in range(first, last):
            action = _actions(cfg, B, k)[team]
            obs, reward, done, _ = env.step(action)
            out.append((obs.clone(), reward.clone(), done.clone(), agent.actions.clone()))
        return out

    run(0, 20)
    snap = env.save_state()
    original = run(20, 60)
    first_obs = env.load_state(snap, resume=True)
    assert torch.equal(first_obs, (base.sim.cam_obs, base.sim.tgt_obs)[team])
    for k, (want, got) in enumerate(zip(original, run(20, 60))):
        for a, b in zip(want, got):
            assert torch.equal(a, b), k
    # branching: the opponent memory of environment d is that of src[d] at save time, the others keep theirs
    snap = env.save_state()
    memory = agent._memory.clone()   # pylint: disable=protected-access
    src = _branch_map(B, 9)
    env.load_state(snap, src=src)
    axis = 2 if kind == 'camera' else 1
    mapped, kept = np.nonzero(src >= 0)[0], np.nonzero(src < 0)[0]
    now = agent._memory   # pylint: disable=protected-access
    pick = lambda t, i: t.index_select(axis, torch.from_numpy(i).cuda())   # noqa: E731
    assert torch.equal(pick(now, mapped), pick(memory, src[mapped]))
    assert torch.equal(pick(now, kept), pick(memory, kept))
    env.close()


@pytest.mark.gpu
def test_refused_snapshots_leave_the_handle_unchanged():
    from mate_b200.sim import BatchedSim

    cfg = _cfg('MATE-4v8-9.yaml')
    B = 256
    sim = BatchedSim(cfg, B, device=0)
    sim.reset(seed=1)
    for k in range(5):
        _step(sim, cfg, k)
    before = sim.save_state()
    other_shape = BatchedSim(_cfg('MATE-4v8-0.yaml'), B, device=0)
    other_shape.reset(seed=1)
    other_cfg = dict(cfg, camera_max_sight_range=cfg['camera_max_sight_range'] + 1.0)
    other_range = BatchedSim(other_cfg, B, device=0)
    other_range.reset(seed=1)
    wrong_version = sim.save_state()
    wrong_version.version += 1
    refused = [
        lambda: sim.load_state(other_shape.save_state()),
        lambda: sim.load_state(other_range.save_state()),
        lambda: sim.load_state(sim.save_state([0, 1, 2])),
        lambda: sim.load_state(before, src=list(range(B)), resume=True),
        lambda: sim.load_state(wrong_version),
    ]
    for case in refused:
        with pytest.raises(ValueError):
            case()
        assert torch.equal(sim.save_state().payload, before.payload)
    for s in (sim, other_shape, other_range):
        s.close()


@pytest.mark.gpu
def test_snapshots_give_back_device_memory():
    from mate_b200.sim import BatchedSim

    cfg = _cfg('MATE-4v8-9.yaml')
    B = 8192

    def one_round():
        sim = BatchedSim(cfg, B, device=0)
        sim.reset(seed=3)
        _step(sim, cfg, 0)
        snap = sim.save_state()
        _step(sim, cfg, 1)
        sim.load_state(snap, resume=True)
        sim.load_state(sim.save_state(list(range(64))), src=np.arange(B) % 64)
        torch.cuda.synchronize()
        sim.close()
        del sim, snap
        gc.collect()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        return torch.cuda.mem_get_info()[0]

    baseline = one_round()   # loads the modules and sets up torch's own state: not a leak
    for k in range(3):
        free = one_round()
        assert abs(free - baseline) <= 2 << 20, (k, free - baseline)
