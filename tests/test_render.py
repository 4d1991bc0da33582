"""rgb_array frames drawn on the GPU (mate_b200_render, DESIGN.md section 7k).

The GPU tests compare the kernel's frames byte for byte with a NumPy restatement of the picture defined in
include/mate_b200.h.  Layer 3 of that restatement (how many cameras see each pixel) is not restated: it is asked of the
simulator's own Camera.perceive, by placing targets at pixel centres in a probe batch and reading mask_ct of an observe
with a transmission draw of 0."""

import ctypes
import os

import numpy as np
import pytest

torch = pytest.importorskip('torch')

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')

V = 1050.0
TERRAIN, OUTSIDE = 0xF4F4F4, 0x404040
WAREHOUSE = (0xE69F00, 0x56B4E9, 0x009E73, 0xCC79A7)
FOV, OBSTACLE, CAMERA, TRACKED, TARGET_EMPTY = 0x0072B2, 0x808080, 0x003E7D, 0xD55E00, 0x202020
ALPHA = 64


# ---------------------------------------------------------------------------------------------- CPU
class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f'the library was called ({name}) although the arguments are refused')


def _recorded_env(reset=True):
    import mate_b200.environment as b200
    from test_communication_wrappers import FilterRecordingSim

    g = np.load(os.path.join(GOLDEN, 'wrappers_4v8-9.npz'))
    base = FilterRecordingSim.make()

    class Sim(base):
        fixture = (g, 'w_')

        def render(self, envs=None, size=800):
            raise AssertionError('the simulator was asked to render although the arguments are refused')

    env = type('MultiAgentTracking', (b200.MultiAgentTracking,), {'_sim_class': Sim})(config=str(g['config_name']), num_envs=1)
    if reset:
        env.reset()
    return env


def test_render_refusals_before_any_library_call():
    import mate_b200.environment as b200

    assert b200.MultiAgentTracking.metadata['render.modes'] == ['rgb_array']
    env = _recorded_env(reset=False)
    with pytest.raises(NotImplementedError, match='rgb_array'):
        env.render()
    with pytest.raises(NotImplementedError, match='rgb_array'):
        env.render(mode='human')
    with pytest.raises(RuntimeError, match='reset'):
        env.render(mode='rgb_array')
    env.reset()
    for size in (15, 4097, 0, -64, 64.0, True, '64', None):
        with pytest.raises(ValueError, match='frame size'):
            env.render(mode='rgb_array', window_size=size)
    for envs in ([1], [-1], [0, 1], [], [[0]], [0.5], np.zeros(0, dtype=np.int64), torch.tensor([2])):
        with pytest.raises(ValueError, match='envs'):
            env.render(mode='rgb_array', window_size=64, envs=envs)


def test_batched_sim_render_checks_its_arguments_first():
    from mate_b200.sim import BatchedSim

    sim = BatchedSim.__new__(BatchedSim)   # the host-side checks only: no device, no handle
    sim.lib, sim.handle, sim.B = _NoLibrary(), None, 4
    for size in (15, 4097, 100.0, False):
        with pytest.raises(ValueError, match='frame size'):
            sim.render(None, size)
    for envs in ([4], [-1], [], [1.0]):
        with pytest.raises(ValueError, match='envs'):
            sim.render(envs, 64)


# ---------------------------------------------------------------------------------------------- NumPy reference
def pixel_centres(S):
    k = np.arange(S, dtype=np.int64)
    x = ((2 * k + 1 - S).astype(np.float64) * V) / S
    y = ((S - 2 * k - 1).astype(np.float64) * V) / S
    return x, y


def _rgb(c):
    return np.array([(c >> 16) & 0xFF, (c >> 8) & 0xFF, c & 0xFF], dtype=np.int64)


def reference_frame(state, e, cfg, S, k_map, tracked):
    """The picture of include/mate_b200.h for environment e of the host state view; k_map [S, S] and tracked [Nt] come
    from the simulator's Camera.perceive."""
    from mate_b200 import constants as consts

    x, y = pixel_centres(S)
    X, Y = np.meshgrid(x, y)
    img = np.where(((np.abs(X) <= 1000.0) & (np.abs(Y) <= 1000.0))[..., None], _rgb(TERRAIN), _rgb(OUTSIDE))
    for w, (wx, wy) in enumerate(consts.WAREHOUSES):
        img[np.maximum(np.abs(X - wx), np.abs(Y - wy)) <= 75.0] = _rgb(WAREHOUSE[w])
    for n in range(int(k_map.max()) if k_map.size else 0):
        m = k_map > n
        img[m] = (img[m] * (255 - ALPHA) + _rgb(FOV) * ALPHA + 127) // 255
    for ox, oy, r in state['obs_xyr'][e]:
        img[(X - ox) * (X - ox) + (Y - oy) * (Y - oy) <= r * r] = _rgb(OBSTACLE)
    cr = float(cfg['camera_radius'])
    for cx, cy in state['cam_xy'][e]:
        img[(X - cx) * (X - cx) + (Y - cy) * (Y - cy) <= cr * cr] = _rgb(CAMERA)
    p = 2.0 * V / S
    r_in, r_out = max(12.0, 1.25 * p), max(22.0, 2.25 * p)
    for t, (tx, ty) in enumerate(state['tgt_xy'][e]):
        d2 = (X - tx) * (X - tx) + (Y - ty) * (Y - ty)
        if tracked[t]:
            img[(d2 > r_in * r_in) & (d2 <= r_out * r_out)] = _rgb(TRACKED)
        goal, weight = state['tgt_goal'][e, t], state['tgt_weight'][e, t]
        img[d2 <= r_in * r_in] = _rgb(WAREHOUSE[goal]) if goal >= 0 and weight > 0 else _rgb(TARGET_EMPTY)
    return img.astype(np.uint8)


class PerceiveProbe:
    """Camera.perceive of the simulator at arbitrary points: a batch of up to 4096 copies of one environment's state,
    each with its targets moved to the points, observed with a transmission draw of 0."""

    def __init__(self, cfg, nt):
        from mate_b200.sim import BatchedSim

        self.nt = nt
        self.P = 4096
        self.sim = BatchedSim(cfg, self.P, device=0)
        self.zeros = np.zeros((self.P, max(int(cfg['num_cameras']), 1), nt), dtype=np.uint8)[:, :int(cfg['num_cameras'])]

    def counts(self, state, e, px, py):
        """Cameras of environment e (of the host view `state`) that see a target at each point (px, py)."""
        base = {name: np.repeat(value[e:e + 1], self.P, axis=0) for name, value in state.items()}
        n = px.size
        out = np.zeros(n, dtype=np.int64)
        per = self.P * self.nt
        for start in range(0, n, per):
            qx, qy = px[start:start + per], py[start:start + per]
            m = qx.size
            xy = base['tgt_xy'].reshape(-1, 2).copy()
            xy[:m, 0], xy[:m, 1] = qx, qy
            arrays = dict(base, tgt_xy=xy.reshape(self.P, self.nt, 2))
            self.sim.set_state(arrays)
            self.sim.observe(replay=(self.zeros, None), aux=True)
            seen = self.sim.aux['mask_ct'].sum(dim=1).reshape(-1).cpu().numpy()
            out[start:start + m] = seen[:m]
        return out

    def tracked(self, state, e):
        return self.counts(state, e, state['tgt_xy'][e, :, 0].copy(), state['tgt_xy'][e, :, 1].copy()) > 0


def expected_frame(probe, state, e, cfg, S):
    x, y = pixel_centres(S)
    X, Y = np.meshgrid(x, y)
    nc = int(cfg['num_cameras'])
    if nc == 0:
        k_map, tracked = np.zeros((S, S), dtype=np.int64), np.zeros(state['tgt_xy'].shape[1], dtype=bool)
    else:
        k_map = probe.counts(state, e, X.reshape(-1), Y.reshape(-1)).reshape(S, S)
        tracked = probe.tracked(state, e)
    return reference_frame(state, e, cfg, S, k_map, tracked), k_map


# ---------------------------------------------------------------------------------------------- GPU
PRESETS = ['MATE-4v8-9.yaml', 'MATE-4v2-9.yaml', 'MATE-8v8-9.yaml', 'MATE-4v8-0.yaml', 'MATE-1v1-9.yaml', 'MATE-Navigation.yaml']


def _sim(preset, B, **overrides):
    from mate_b200.config import flatten_config, read_config
    from mate_b200.sim import BatchedSim

    cfg = flatten_config(read_config(preset, **overrides))
    return cfg, BatchedSim(cfg, B, device=0)


def _actions(cfg, B, k):
    gen = torch.Generator(device='cuda')
    gen.manual_seed(3000 + k)
    scale = torch.tensor([cfg['camera_rotation_step'], cfg['camera_zooming_step']], device='cuda')
    cam = (torch.rand((B, max(cfg['num_cameras'], 1), 2), device='cuda', generator=gen) * 2 - 1) * scale
    tgt = (torch.rand((B, cfg['num_targets'], 2), device='cuda', generator=gen) * 2 - 1) * cfg['target_step_size']
    return cam[:, :cfg['num_cameras']].contiguous(), tgt


def _run(sim, cfg, steps, first=0):
    for k in range(first, first + steps):
        sim.step(*_actions(cfg, sim.B, k), auto_reset=True)


@pytest.mark.gpu
@pytest.mark.parametrize('preset', PRESETS)
def test_frames_match_the_reference(preset):
    B = 48
    cfg, sim = _sim(preset, B)
    probe = PerceiveProbe(cfg, int(cfg['num_targets']))
    sim.reset(seed=11)
    fov_pixels = 0
    for phase in ('reset', 'steps'):
        if phase == 'steps':
            _run(sim, cfg, 50)
        torch.cuda.synchronize()
        state = sim.get_state()
        for e in (0, 17, B - 1):
            for S in (64, 256):
                frame = sim.render([e], size=S)[0].cpu().numpy()
                want, k_map = expected_frame(probe, state, e, cfg, S)
                fov_pixels += int((k_map > 0).sum())
                bad = np.argwhere((frame != want).any(-1))
                assert bad.size == 0, (preset, phase, e, S, len(bad), bad[:5].tolist(),
                                       [(frame[i, j].tolist(), want[i, j].tolist(), int(k_map[i, j])) for i, j in bad[:5]])
    if cfg['num_cameras'] > 0:
        assert fov_pixels > 0, preset   # the fields of view are in the picture
    if preset == 'MATE-4v8-9.yaml':   # one large frame
        frame = sim.render([B - 1], size=1024)[0].cpu().numpy()
        want, _ = expected_frame(probe, state, B - 1, cfg, 1024)
        assert np.array_equal(frame, want)


@pytest.mark.gpu
def test_frame_sizes_that_are_not_multiples_of_four():
    """Sizes whose rows are not whole 32-bit words take the byte stores; the picture is the same."""
    B = 8
    cfg, sim = _sim('MATE-4v8-9.yaml', B)
    probe = PerceiveProbe(cfg, int(cfg['num_targets']))
    sim.reset(seed=5)
    _run(sim, cfg, 10)
    torch.cuda.synchronize()
    state = sim.get_state()
    for S in (16, 61, 130):
        frames = sim.render([B - 1, 2], size=S).cpu().numpy()
        for i, e in enumerate((B - 1, 2)):
            want, _ = expected_frame(probe, state, e, cfg, S)
            assert np.array_equal(frames[i], want), S


@pytest.mark.gpu
@pytest.mark.parametrize('preset', ['MATE-4v8-9.yaml', 'MATE-8v8-9.yaml'])
def test_a_frame_is_a_function_of_the_state(preset, monkeypatch):
    from mate_b200 import _abi
    from mate_b200.sim import BatchedSim

    B, S = 40, 128
    cfg, sim = _sim(preset, B, max_episode_steps=7)
    sim.reset(seed=3)
    _run(sim, cfg, 20)
    want = sim.render(None, size=S)
    e = 13
    alone = sim.render([e], size=S)[0]
    mixed = sim.render(torch.tensor([e, 0, e, B - 1, e], device='cuda'), size=S)
    assert torch.equal(alone, want[e]) and all(torch.equal(mixed[i], alone) for i in (0, 2, 4))
    assert torch.equal(mixed[1], want[0]) and torch.equal(mixed[3], want[B - 1])
    snapshot = sim.save_state()
    # another batch size, branched from e; float16 rows; single-team rows
    other = BatchedSim(cfg, 300, device=0)
    other.load_state(snapshot, src=[e] * 300)
    assert torch.equal(other.render([0, 299], size=S)[1], alone)
    for kwargs in ({'observation_dtype': torch.float16}, {'observed_team': 'camera'}, {'observed_team': 'target'}):
        twin = BatchedSim(cfg, B, device=0, **kwargs)
        twin.load_state(snapshot)
        twin.observe()
        assert torch.equal(twin.render(size=S), want), kwargs
    # registered observation wrappers on both folded paths
    for fold in ('1', '0'):
        monkeypatch.setenv('MATE_B200_FOLD', fold)
        twin = BatchedSim(cfg, B, device=0)
        twin.load_state(snapshot)
        twin.set_observation_wrappers([_abi.OBS_ENHANCED_CAMERA, _abi.OBS_RELATIVE, _abi.OBS_RESCALED])
        twin.observe()
        assert torch.equal(twin.render(size=S), want), fold
    monkeypatch.delenv('MATE_B200_FOLD')
    # both refill modes, with auto-resets on the way: the same states give the same frames
    frames = []
    for refill in ('sync', None):
        if refill is None:
            monkeypatch.delenv('MATE_B200_REFILL', raising=False)
        else:
            monkeypatch.setenv('MATE_B200_REFILL', refill)
        _, twin = _sim(preset, B, max_episode_steps=7)
        twin.reset(seed=3)
        _run(twin, cfg, 20)
        frames.append(twin.render(size=S))
    assert torch.equal(frames[0], want) and torch.equal(frames[1], want)


def _aux_bits(sim):
    return {k: v.clone() for k, v in sim.aux.items()}


@pytest.mark.gpu
def test_rendering_changes_nothing():
    B = 64
    cfg, a = _sim('MATE-4v8-9.yaml', B, max_episode_steps=30)
    _, b = _sim('MATE-4v8-9.yaml', B, max_episode_steps=30)
    a.reset(seed=21)
    b.reset(seed=21)
    before = a.save_state().payload.clone()
    a.render(None, size=96)
    a.render([5, 5, 63], size=33)
    torch.cuda.synchronize()
    assert torch.equal(a.save_state().payload, before)
    for k in range(200):
        cam, tgt = _actions(cfg, B, k)
        a.step(cam, tgt, auto_reset=True, aux=True)
        a.render(torch.arange(0, B, 3, device='cuda', dtype=torch.int32), size=48)
        b.step(cam, tgt, auto_reset=True, aux=True)
        assert torch.equal(a.cam_obs.view(torch.int32), b.cam_obs.view(torch.int32)), k
        assert torch.equal(a.tgt_obs.view(torch.int32), b.tgt_obs.view(torch.int32)), k
        assert torch.equal(a.rewards, b.rewards) and torch.equal(a.done, b.done), k
        for key, value in a.aux.items():
            assert torch.equal(value, b.aux[key]), (k, key)
    assert int(a.episode_stats()[0].item()) > 0   # episodes ended and were reset on the way


@pytest.mark.gpu
def test_device_index_maps_streams_and_refusals():
    B, S = 12, 64
    cfg, sim = _sim('MATE-4v8-9.yaml', B)
    sim.reset(seed=4)
    _run(sim, cfg, 5)
    want = sim.render(None, size=S)
    out = torch.full((5, S, S, 3), 0xA5, dtype=torch.uint8, device='cuda')
    env = torch.tensor([3, -1, B, 1 << 30, B - 1], dtype=torch.int32, device='cuda')
    rc = sim.lib.mate_b200_render(sim.handle, ctypes.c_void_p(env.data_ptr()), 5, S, ctypes.c_void_p(out.data_ptr()),
                                  ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(out[0], want[3]) and torch.equal(out[4], want[B - 1])
    assert bool((out[1:4] == 0xA5).all())   # out-of-range entries: frames unwritten
    assert torch.equal(sim.render(torch.tensor([B, 2], device='cuda'), size=S)[1], want[2])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        frames = sim.render([7, 0], size=S)
    side.synchronize()
    assert torch.equal(frames[0], want[7]) and torch.equal(frames[1], want[0])
    # the C ABI's refusals (MATE_EINVAL before any launch)
    ptr, stream = ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(0)
    launches = sim.launch_count
    for args in ((None, B - 1, S, ptr), (ctypes.c_void_p(env.data_ptr()), 0, S, ptr),
                 (ctypes.c_void_p(env.data_ptr()), -1, S, ptr), (None, B, 15, ptr), (None, B, 4097, ptr), (None, B, S, None)):
        assert sim.lib.mate_b200_render(sim.handle, *args, stream) == -1, args
    assert sim.lib.mate_b200_render(None, None, B, S, ptr, stream) == -1
    assert sim.launch_count == launches


@pytest.mark.gpu
def test_environment_render():
    import mate_b200

    single = mate_b200.MultiAgentTracking('MATE-4v8-9.yaml')
    with pytest.raises(RuntimeError, match='reset'):
        single.render('rgb_array')
    single.reset(seed=9)
    for _ in range(3):
        single.step((np.full((4, 2), 0.5), np.full((8, 2), 3.0)))
    frame = single.render('rgb_array', window_size=200)
    assert isinstance(frame, np.ndarray) and frame.dtype == np.uint8 and frame.shape == (200, 200, 3)
    batched = mate_b200.MultiAgentTracking('MATE-4v8-9.yaml', num_envs=6)
    batched.reset(seed=1)
    batched.sim.load_state(single.sim.save_state(), src=[0] * 6)
    frames = batched.render('rgb_array', window_size=200)
    assert frames.is_cuda and frames.dtype == torch.uint8 and tuple(frames.shape) == (1, 200, 200, 3)
    assert np.array_equal(frames[0].cpu().numpy(), frame)
    assert tuple(batched.render(mode='rgb_array', window_size=64, envs=[5, 0, 5]).shape) == (3, 64, 64, 3)
    with pytest.raises(NotImplementedError, match='rgb_array'):
        batched.render()

    # the README's MultiCamera stack forwards render through its wrappers
    env = mate_b200.make('MATE-4v8-9-v0', num_envs=16, wrappers=[
        mate_b200.MoreTrainingInformation, mate_b200.RepeatedRewardIndividualDone,
        lambda e: mate_b200.AuxiliaryCameraRewards(e, coefficients={'raw_reward': 1.0, 'coverage_rate': 1.0}, reduction='mean'),
        lambda e: mate_b200.MultiCamera(e, target_agent=mate_b200.GreedyTargetAgent(seed=0))])
    env.reset(seed=2)
    video = []
    for k in range(4):
        nc = env.unwrapped.num_cameras
        env.step(torch.zeros((16, nc, 2), device='cuda'))
        video.append(env.render(mode='rgb_array', window_size=64, envs=range(0, 16, 4)))
    video = torch.stack(video, dim=1)
    assert tuple(video.shape) == (4, 4, 64, 64, 3)
    assert torch.equal(video[:, -1], env.unwrapped.sim.render([0, 4, 8, 12], size=64))
