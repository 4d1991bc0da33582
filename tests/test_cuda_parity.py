"""GPU parity tests (run with ``-m gpu`` on the B200 box): the CUDA path, called through the
C ABI, against (a) the committed traces of the unmodified reference and (b) the C oracle on
seeded batched inputs.

Tolerances (BASELINE.json north_star): visibility masks, cargo counts, rewards and done
flags bit-exact; positions / orientations / observations within 1e-5 relative (fp32 I/O)."""

import numpy as np
import pytest

import golden_util as gu

torch = pytest.importorskip('torch')
pytestmark = pytest.mark.gpu

OBS_RTOL, OBS_ATOL = 1e-5, 1e-5


def _sim(cfg, B):
    from mate_b200.sim import BatchedSim

    return BatchedSim(cfg, B, device=0)


def _np(t):
    return t.detach().cpu().numpy()


@pytest.mark.parametrize('name', gu.trace_names())
def test_golden_trace(name):
    """Replay a recorded episode of the UNMODIFIED reference through the CUDA kernel."""
    g = gu.load(name)
    cfg = gu.flat_config(g)
    nc = cfg['num_cameras']
    sim = _sim(cfg, 1)
    sim.set_state(gu.state_arrays(g))
    aux = sim.alloc_aux()
    cam0, tgt0 = sim.observe(replay=(g['init_transmit'][None], None), aux=True)
    if nc:
        np.testing.assert_allclose(_np(cam0)[0], g['init_cam_obs'], rtol=OBS_RTOL, atol=OBS_ATOL)
    np.testing.assert_allclose(_np(tgt0)[0], g['init_tgt_obs'], rtol=OBS_RTOL, atol=OBS_ATOL)
    for key in ('mask_ct', 'mask_cc', 'mask_co', 'mask_tc', 'mask_to', 'mask_tt'):
        assert (_np(aux[key])[0] == g['init_' + key]).all(), key

    T = int(g['num_steps'])
    obs_steps = {int(s): i for i, s in enumerate(g['obs_steps'])}
    tangent_flips = 0
    cam_act = torch.from_numpy(g['step_cam_act'].astype(np.float32)).cuda()
    tgt_act = torch.from_numpy(g['step_tgt_act'].astype(np.float32)).cuda()
    for k in range(T):
        (cam, tgt), rewards, done = sim.step(
            cam_act[k][None], tgt_act[k][None], auto_reset=False,
            replay=(g['step_transmit'][k][None], g['step_goal_choice'][k][None]), aux=True)
        ctx = f'{name} step {k}'
        mask_ct = _np(aux['mask_ct'])[0]
        if not (mask_ct == g['step_mask_ct'][k]).all():
            for c, t in np.argwhere(mask_ct != g['step_mask_ct'][k]):
                assert gu.in_tangent_sliver(g['init_cam_xy'][c], g['step_tgt_xy'][k][t], g['init_obs_xyr'],
                                            cfg['camera_max_sight_range']), (ctx, c, t)
                tangent_flips += 1
            sim.set_state(gu.step_state_arrays(g, k))
            continue
        rew = _np(rewards)[0]
        assert rew[0] == g['step_reward'][k, 0] and rew[1] == g['step_reward'][k, 1], ctx
        assert bool(_np(done)[0]) == bool(g['step_done'][k]), ctx
        for key in ('mask_cc', 'mask_tc', 'mask_to', 'mask_tt'):
            assert (_np(aux[key])[0] == g['step_' + key][k]).all(), (ctx, key)
        assert (_np(aux['target_dones'])[0] == g['step_target_dones'][k]).all(), ctx
        assert (_np(aux['is_colliding'])[0] == g['step_tgt_colliding'][k]).all(), ctx
        assert _np(aux['num_delivered'])[0] == g['step_num_delivered'][k], ctx
        np.testing.assert_allclose(_np(aux['coverage'])[0], g['step_coverage'][k], rtol=1e-5, atol=1e-6, err_msg=ctx)
        np.testing.assert_allclose(_np(aux['warehouse_dist'])[0], g['step_warehouse_dist'][k], rtol=1e-5, err_msg=ctx)
        if k in obs_steps:
            i = obs_steps[k]
            if nc:
                np.testing.assert_allclose(_np(cam)[0], g['step_cam_obs'][i], rtol=OBS_RTOL, atol=OBS_ATOL, err_msg=ctx)
            np.testing.assert_allclose(_np(tgt)[0], g['step_tgt_obs'][i], rtol=OBS_RTOL, atol=OBS_ATOL, err_msg=ctx)
        if k % 200 == 0 or k == T - 1:
            st = sim.get_state()
            np.testing.assert_allclose(st['tgt_xy'][0], g['step_tgt_xy'][k], rtol=0, atol=1e-8, err_msg=ctx)
            np.testing.assert_allclose(st['cam_phi'][0], g['step_cam_phi'][k], rtol=0, atol=1e-9, err_msg=ctx)
            np.testing.assert_allclose(st['cam_theta'][0], g['step_cam_theta'][k], rtol=0, atol=1e-9, err_msg=ctx)
            assert (st['tgt_goal'][0] == g['step_tgt_goal'][k]).all(), ctx
            assert (st['tgt_weight'][0] == g['step_tgt_goal_weight'][k]).all(), ctx
            assert (st['tgt_bounty'][0] == g['step_bounties'][k]).all(), ctx
            assert (st['tgt_empty_bits'][0] == gu.empty_bits_to_int(g['step_tgt_empty_bits'][k])).all(), ctx
            assert (st['remaining'][0] == g['step_remaining'][k]).all(), ctx
            assert (st['awaiting'][0] == g['step_awaiting'][k]).all(), ctx
            assert st['episode_step'][0] == g['step_episode_step'][k], ctx
            assert st['episode_reward'][0, 0] == g['step_ep_reward'][k], ctx
            assert st['episode_reward'][0, 1] == g['step_delayed_ep_reward'][k], ctx
    assert tangent_flips <= max(2, T // 2000), tangent_flips


@pytest.mark.parametrize('name', gu.reset_names())
def test_reference_reset_states(name):
    """First observation + masks for several reference resets (on-the-fly FOV vs the
    reference's materialised polyline)."""
    g = gu.load(name)
    cfg = gu.flat_config(g)
    nc = cfg['num_cameras']
    count = int(g['count'])
    sim = _sim(cfg, count)
    sim.set_state(gu.stack_states([gu.state_arrays(g, 'reset_', i) for i in range(count)]))
    aux = sim.alloc_aux()
    cam, tgt = sim.observe(replay=(g['reset_transmit'], None), aux=True)
    if nc:
        np.testing.assert_allclose(_np(cam), g['reset_cam_obs'], rtol=OBS_RTOL, atol=OBS_ATOL)
    np.testing.assert_allclose(_np(tgt), g['reset_tgt_obs'], rtol=OBS_RTOL, atol=OBS_ATOL)
    for key in ('mask_ct', 'mask_cc', 'mask_co', 'mask_tc', 'mask_to', 'mask_tt'):
        assert (_np(aux[key]) == g['reset_' + key]).all(), key


def _goal_seeking_actions(rng, cfg, state, B, noise=0.3):
    """fp32 joint actions: targets head for their goal warehouse (so cargo gets delivered),
    cameras turn randomly."""
    nc, nt = cfg['num_cameras'], cfg['num_targets']
    wh = 925.0 * np.array([[1.0, 1.0], [-1.0, 1.0], [-1.0, -1.0], [1.0, -1.0]])
    goal = state['tgt_goal']
    dest = wh[np.where(goal >= 0, goal, rng.randint(0, 4, size=goal.shape))]
    direction = dest - state['tgt_xy']
    direction /= np.maximum(np.linalg.norm(direction, axis=-1, keepdims=True), 1e-9)
    tgt_act = cfg['target_step_size'] * (direction + noise * rng.uniform(-1, 1, size=direction.shape))
    cam_act = rng.uniform(-1, 1, size=(B, nc, 2)) * np.array([cfg['camera_rotation_step'], cfg['camera_zooming_step']])
    return cam_act.astype(np.float32), tgt_act.astype(np.float32)


CASES = [
    # preset, B, steps, overrides[, warp tile (MATE_B200_TILE)]; every compiled shape (tests/test_shape_matrix.py)
    ('MATE-4v8-9.yaml', 512, 160, {}),
    ('MATE-4v8-9.yaml', 256, 120, {'max_episode_steps': 37}),      # time-limit done + auto-reset
    ('MATE-8v8-9.yaml', 256, 100, {}),
    ('MATE-4v2-9.yaml', 509, 120, {}),                             # ragged tail (B % envs-per-CTA != 0)
    ('MATE-4v8-0.yaml', 256, 100, {}),
    ('MATE-Navigation.yaml', 256, 150, {}),
    ('MATE-2v4-9.yaml', 130, 100, {'max_episode_steps': 51}),
    ('MATE-1v1-9.yaml', 200, 100, {}),
    ('MATE-4v4-0.yaml', 64, 60, {}),
    ('MATE-1v1-0.yaml', 203, 90, {'max_episode_steps': 29}),
    ('MATE-1v2-0.yaml', 157, 90, {}),                              # camera rows of 39 floats: scalar stores
    ('MATE-1v2-9.yaml', 131, 90, {'max_episode_steps': 41}),       # camera rows of 75 floats: scalar stores
    ('MATE-2v2-0.yaml', 99, 90, {'max_episode_steps': 33}),        # 4-float camera / 2-float target stores
    ('MATE-2v2-9.yaml', 173, 90, {}),
    ('MATE-2v4-0.yaml', 117, 90, {'max_episode_steps': 43}),
    ('MATE-4v2-0.yaml', 101, 90, {}),
    ('MATE-4v4-9.yaml', 141, 90, {'max_episode_steps': 39}),       # dense block copy, all three obstacle-round classes
    ('MATE-8v8-0.yaml', 67, 80, {}),
    # the odd-row shapes again in the warp tiles of large batches: below 8192 environments the step runs in tiles of 8
    # (mate_sim_create), so every case above does, and MATE_B200_TILE picks 32 (from 24 576 environments on) or 16 here
    ('MATE-1v1-0.yaml', 77, 60, {'max_episode_steps': 23}, 32),
    ('MATE-1v2-0.yaml', 45, 60, {}, 32),
    ('MATE-1v2-9.yaml', 53, 60, {'max_episode_steps': 27}, 32),
    ('MATE-2v2-0.yaml', 39, 60, {}, 32),
    ('MATE-2v2-9.yaml', 61, 60, {'max_episode_steps': 25}, 32),
    ('MATE-1v2-9.yaml', 83, 60, {}, 16),
    ('MATE-2v2-0.yaml', 71, 60, {'max_episode_steps': 31}, 16),
]
# the ids of the cases without a tile stay those pytest gave the four-field tuples
CASE_PARAMS = [case if len(case) == 5 else case + (None,) for case in CASES]
CASE_IDS = [f'{p}-{b}-{s}-overrides{i}' + (f'-tile{tile}' if tile else '') for i, (p, b, s, _, tile) in enumerate(CASE_PARAMS)]


@pytest.mark.parametrize('preset,B,steps,overrides,tile', CASE_PARAMS, ids=CASE_IDS)
def test_cuda_vs_oracle(preset, B, steps, overrides, tile, monkeypatch):
    """Reset + step + auto-reset on the GPU against the float64 C oracle, same Philox streams."""
    from mate_b200.config import flatten_config, read_config
    from oracle.oracle import Oracle

    if tile:
        monkeypatch.setenv('MATE_B200_TILE', str(tile))
    cfg = flatten_config(read_config(preset, **overrides))
    nc = cfg['num_cameras']
    seed = 1234
    sim = _sim(cfg, B)
    ref = Oracle(cfg, B, num_threads=8)
    cam0, tgt0 = sim.reset(seed=seed)
    rcam0, rtgt0 = ref.reset(seed=seed)
    s_cuda, s_ref = sim.get_state(), ref.get_state()
    for key in s_ref:
        if s_ref[key].dtype.kind == 'f':
            np.testing.assert_allclose(s_cuda[key], s_ref[key], rtol=0, atol=1e-9, err_msg=key)
        else:
            assert (s_cuda[key] == s_ref[key]).all(), key
    if nc:
        np.testing.assert_allclose(_np(cam0), rcam0, rtol=OBS_RTOL, atol=OBS_ATOL)
    np.testing.assert_allclose(_np(tgt0), rtgt0, rtol=OBS_RTOL, atol=OBS_ATOL)

    rng = np.random.RandomState(99)
    aux = sim.alloc_aux()
    raux = ref.alloc_aux()
    total_done = 0
    total_delivered = 0
    for k in range(steps):
        state = ref.get_state()
        if k % 3 == 2:   # some purely random steps as well
            cam_act = (rng.uniform(-1, 1, (B, nc, 2)) * [cfg['camera_rotation_step'], cfg['camera_zooming_step']]).astype(np.float32)
            tgt_act = (rng.uniform(-1, 1, (B, cfg['num_targets'], 2)) * cfg['target_step_size']).astype(np.float32)
        else:
            cam_act, tgt_act = _goal_seeking_actions(rng, cfg, state, B)
        (cam, tgt), rew, done = sim.step(torch.from_numpy(cam_act).cuda(), torch.from_numpy(tgt_act).cuda(),
                                         auto_reset=True, aux=True)
        (rcam, rtgt), rrew, rdone = ref.step(cam_act, tgt_act, seed=seed, auto_reset=True, aux=raux)
        ctx = f'{preset} step {k}'
        for key in ('mask_ct', 'mask_cc', 'mask_co', 'mask_tc', 'mask_to', 'mask_tt', 'target_dones',
                    'is_colliding', 'num_delivered', 'episode_step'):
            assert (_np(aux[key]) == raux[key]).all(), (ctx, key)
        assert (_np(rew) == rrew).all(), ctx
        assert (_np(done) == rdone).all(), ctx
        np.testing.assert_allclose(_np(aux['coverage']), raux['coverage'], rtol=1e-6, atol=1e-7, err_msg=ctx)
        np.testing.assert_allclose(_np(aux['warehouse_dist']), raux['warehouse_dist'], rtol=1e-6, err_msg=ctx)
        if nc:
            np.testing.assert_allclose(_np(cam), rcam, rtol=OBS_RTOL, atol=OBS_ATOL, err_msg=ctx)
        np.testing.assert_allclose(_np(tgt), rtgt, rtol=OBS_RTOL, atol=OBS_ATOL, err_msg=ctx)
        total_done += int(rdone.sum())
        total_delivered = max(total_delivered, int(raux['num_delivered'].max()))
        if k % 20 == 19 or k == steps - 1:
            s_cuda, s_ref = sim.get_state(), ref.get_state()
            for key in s_ref:
                if s_ref[key].dtype.kind == 'f':
                    np.testing.assert_allclose(s_cuda[key], s_ref[key], rtol=0, atol=1e-8, err_msg=(ctx, key))
                else:
                    assert (s_cuda[key] == s_ref[key]).all(), (ctx, key)
    if 'max_episode_steps' in overrides:
        assert total_done >= B, 'the time-limit auto-reset was not exercised'
    stats = _np(sim.episode_stats())
    rstats = ref.episode_stats()
    np.testing.assert_allclose(stats[:6], rstats[:6], rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize('mode', ['1', '2'])   # 2: only the calls that patch changes take the compacted leg, the others copy densely
def test_step_host_rows_kept(mode, monkeypatch):
    """MATE_STEP_HOST_ROWS_KEPT: with the caller's buffers reused and untouched between calls only the 64-byte groups
    that differ from the previous call's rows cross the link and are rewritten; the buffers still equal the rows of the
    device-resident step (auto-resets every 4 steps change many entries at once).  A call without the flag rewrites
    everything: garbage the caller left in the buffers is gone afterwards; so does a call with other buffers."""
    from mate_b200.config import flatten_config, read_config

    monkeypatch.setenv('MATE_B200_HOST_COMPACT', mode)
    monkeypatch.setenv('MATE_B200_REFILL', 'sync')
    cfg = flatten_config(read_config('MATE-4v8-9.yaml', max_episode_steps=4))
    B = 2048
    a, b = _sim(cfg, B), _sim(cfg, B)
    a.reset(seed=9)
    b.reset(seed=9)
    rng = np.random.RandomState(3)

    def buffers():
        return (torch.zeros((B, 4, a.dc)).pin_memory(), torch.zeros((B, 8, a.dt)).pin_memory(),
                torch.zeros((B, 2)).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory())

    out, other = buffers(), buffers()
    for k in range(14):
        cam_act = torch.from_numpy((rng.uniform(-1, 1, (B, 4, 2)) * [5.0, 2.5]).astype(np.float32)).pin_memory()
        tgt_act = torch.from_numpy((rng.uniform(-1, 1, (B, 8, 2)) * 20.0).astype(np.float32)).pin_memory()
        (cam, tgt), rew, done = a.step(cam_act.cuda(), tgt_act.cuda(), auto_reset=True)
        if k == 6:     # the caller scribbles over the buffers and says so by not passing the flag
            out[0].fill_(7.0); out[1].fill_(-3.0)
            b.step_host(cam_act, tgt_act, out, auto_reset=True, rows_kept=False)
        elif k == 10:  # other buffers (all 5.0): the flag is passed wrongly, the library notices the new addresses
            other[0].fill_(5.0); other[1].fill_(5.0)
            out, other = other, out
            b.step_host(cam_act, tgt_act, out, auto_reset=True, rows_kept=True)
        else:
            b.step_host(cam_act, tgt_act, out, auto_reset=True, rows_kept=True)
        torch.cuda.synchronize()
        assert torch.equal(cam.cpu(), out[0]) and torch.equal(tgt.cpu(), out[1]), k
        assert torch.equal(rew.cpu(), out[2]) and torch.equal(done.cpu(), out[3]), k


@pytest.mark.parametrize('mode', ['0', '1', '2'])
@pytest.mark.parametrize('preset', ['MATE-Navigation.yaml', 'MATE-8v8-9.yaml', 'MATE-4v2-9.yaml', 'MATE-4v8-0.yaml'])
def test_step_host_other_shapes(preset, mode, monkeypatch):
    """Every device -> host leg of mate_b200_step_host on the other BASELINE shapes (no cameras; 8 cameras; rows that are
    not whole 16-byte chunks and therefore always copied densely; no obstacles): the caller's buffers equal the rows of
    the device-resident step, with and without MATE_STEP_HOST_ROWS_KEPT."""
    from mate_b200.config import flatten_config, read_config

    monkeypatch.setenv('MATE_B200_HOST_COMPACT', mode)
    monkeypatch.setenv('MATE_B200_REFILL', 'sync')
    cfg = flatten_config(read_config(preset, max_episode_steps=5))
    nc, nt = cfg['num_cameras'], cfg['num_targets']
    B = 1536
    a, b = _sim(cfg, B), _sim(cfg, B)
    a.reset(seed=3)
    b.reset(seed=3)
    out = (torch.zeros((B, max(nc, 1), a.dc)).pin_memory(), torch.zeros((B, nt, a.dt)).pin_memory(),
           torch.zeros((B, 2)).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory())
    rng = np.random.RandomState(0)
    legs = set()
    for k in range(8):
        cam_act = torch.from_numpy((rng.uniform(-1, 1, (B, max(nc, 1), 2)) * [5.0, 2.5]).astype(np.float32)).pin_memory()
        tgt_act = torch.from_numpy((rng.uniform(-1, 1, (B, nt, 2)) * 20.0).astype(np.float32)).pin_memory()
        (cam, tgt), rew, done = a.step(cam_act.cuda(), tgt_act.cuda(), auto_reset=True)
        b.step_host(cam_act, tgt_act, out, auto_reset=True, rows_kept=(k != 3))
        torch.cuda.synchronize()
        legs.add(b.host_leg_info()[0])
        if nc:
            assert torch.equal(cam.cpu(), out[0]), k
        assert torch.equal(tgt.cpu(), out[1]) and torch.equal(rew.cpu(), out[2]) and torch.equal(done.cpu(), out[3]), k
    whole_chunks = (4 * nc * a.dc) % 16 == 0 and (4 * nt * a.dt) % 16 == 0
    expected = {'0': {0}, '1': {1, 2}, '2': {0, 2}}[mode] if whole_chunks else {0}
    assert legs == expected, legs


@pytest.mark.parametrize('compact', ['0', '1'])
def test_step_host_matches_device_step(compact, monkeypatch):
    """Both device -> host legs of mate_b200_step_host (dense copy; compacted rows expanded by host threads,
    mate_hostpath.cuh) hand the caller exactly the bytes of the device-resident step."""
    from mate_b200.config import flatten_config, read_config

    monkeypatch.setenv('MATE_B200_HOST_COMPACT', compact)
    cfg = flatten_config(read_config('MATE-4v8-9.yaml'))
    B = 1024
    a, b = _sim(cfg, B), _sim(cfg, B)
    a.reset(seed=5)
    b.reset(seed=5)
    rng = np.random.RandomState(1)
    out = (torch.zeros((B, 4, a.dc)).pin_memory(), torch.zeros((B, 8, a.dt)).pin_memory(),
           torch.zeros((B, 2)).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory())
    for _ in range(5):
        cam_act = torch.from_numpy((rng.uniform(-1, 1, (B, 4, 2)) * [5.0, 2.5]).astype(np.float32)).pin_memory()
        tgt_act = torch.from_numpy((rng.uniform(-1, 1, (B, 8, 2)) * 20.0).astype(np.float32)).pin_memory()
        (cam, tgt), rew, done = a.step(cam_act.cuda(), tgt_act.cuda())
        b.step_host(cam_act, tgt_act, out)
        torch.cuda.synchronize()
        assert torch.equal(cam.cpu(), out[0]) and torch.equal(tgt.cpu(), out[1])
        assert torch.equal(rew.cpu(), out[2]) and torch.equal(done.cpu(), out[3])


def test_step_host_adopts_prepared_resets(monkeypatch):
    """The host-buffer path launches the step in chunks; its auto-resets adopt the prepared next episodes like the
    device path (round 1 dropped them for every chunk and never refilled) and give the same results."""
    from mate_b200.config import flatten_config, read_config

    cfg = flatten_config(read_config('MATE-4v8-9.yaml', max_episode_steps=4))
    B = 4096
    monkeypatch.setenv('MATE_B200_REFILL', 'sync')
    a, b = _sim(cfg, B), _sim(cfg, B)
    a.reset(seed=5)
    b.reset(seed=5)
    rng = np.random.RandomState(1)
    out = (torch.zeros((B, 4, a.dc)).pin_memory(), torch.zeros((B, 8, a.dt)).pin_memory(),
           torch.zeros((B, 2)).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory())
    for k in range(12):
        cam_act = torch.from_numpy((rng.uniform(-1, 1, (B, 4, 2)) * [5.0, 2.5]).astype(np.float32)).pin_memory()
        tgt_act = torch.from_numpy((rng.uniform(-1, 1, (B, 8, 2)) * 20.0).astype(np.float32)).pin_memory()
        (cam, tgt), rew, done = a.step(cam_act.cuda(), tgt_act.cuda(), auto_reset=True)
        b.step_host(cam_act, tgt_act, out, auto_reset=True)
        torch.cuda.synchronize()
        assert torch.equal(cam.cpu(), out[0]) and torch.equal(tgt.cpu(), out[1]), k
        assert torch.equal(rew.cpu(), out[2]) and torch.equal(done.cpu(), out[3]), k
    stats_a, stats_b = _np(a.episode_stats()), _np(b.episode_stats())
    assert stats_b[0] == stats_a[0] >= 2 * B
    assert stats_b[6] == stats_b[0] and stats_b[7] == 0, stats_b[:8]   # every reset of the host path adopted a prepared episode


@pytest.mark.parametrize('preset,overrides', [('MATE-4v8-9.yaml', {'max_episode_steps': 9}),
                                              ('MATE-Navigation.yaml', {'max_episode_steps': 7}),
                                              ('MATE-2v4-9.yaml', {'max_episode_steps': 1})])
def test_prepared_resets_equal_resets_in_place(preset, overrides, monkeypatch):
    """Auto-reset through the prepared next-episode state (MATE_B200_REFILL=sync: prepared after every
    step, so always adopted) gives bit-identical observations, rewards, done flags and state to the reset
    computed in place (MATE_B200_REFILL=0), and both paths are really taken."""
    from mate_b200.config import flatten_config, read_config

    cfg = flatten_config(read_config(preset, **overrides))
    nc, nt = cfg['num_cameras'], cfg['num_targets']
    B = 200
    monkeypatch.setenv('MATE_B200_REFILL', 'sync')
    a = _sim(cfg, B)
    monkeypatch.setenv('MATE_B200_REFILL', '0')
    b = _sim(cfg, B)
    a.reset(seed=11)
    b.reset(seed=11)
    rng = np.random.RandomState(3)
    for k in range(40):
        cam_act = torch.from_numpy((rng.uniform(-1, 1, (B, nc, 2)) * [cfg['camera_rotation_step'], cfg['camera_zooming_step']]).astype(np.float32)).cuda()
        tgt_act = torch.from_numpy((rng.uniform(-1, 1, (B, nt, 2)) * cfg['target_step_size']).astype(np.float32)).cuda()
        (cam_a, tgt_a), rew_a, done_a = a.step(cam_act, tgt_act, auto_reset=True)
        (cam_b, tgt_b), rew_b, done_b = b.step(cam_act, tgt_act, auto_reset=True)
        assert torch.equal(tgt_a, tgt_b) and torch.equal(rew_a, rew_b) and torch.equal(done_a, done_b), k
        if nc:
            assert torch.equal(cam_a, cam_b), k
    sa, sb = a.get_state(), b.get_state()
    for key in sa:
        assert (sa[key] == sb[key]).all(), key
    stats_a, stats_b = _np(a.episode_stats()), _np(b.episode_stats())
    assert stats_a[0] == stats_b[0] > 0
    if overrides['max_episode_steps'] > 1:
        assert stats_a[6] == stats_a[0] and stats_a[7] == 0      # every reset adopted the prepared state
    else:
        assert stats_a[6] + stats_a[7] == stats_a[0] and stats_a[6] > 0   # two-step episodes: both paths, same results
    assert stats_b[7] == stats_b[0] and stats_b[6] == 0          # every reset computed in place


def test_async_refill_equals_resets_in_place(monkeypatch):
    """The mode bench.py times: prepared episodes refilled by a MODE_PREPARE launch on the SIDE stream every few
    steps, racing with the step launches of the main stream (no synchronisation between them but the release /
    acquire of the per-environment `ready` tag).  Whatever an auto-reset finds -- a ready prepared episode or a
    stale tag -- the results are bit-identical to resets computed in place, and both paths occur."""
    from mate_b200.config import flatten_config, read_config

    cfg = flatten_config(read_config('MATE-4v8-9.yaml', max_episode_steps=5))
    nc, nt = cfg['num_cameras'], cfg['num_targets']
    B = 8192
    monkeypatch.setenv('MATE_B200_REFILL', '16')    # side stream, every 16 steps: an episode of 6 steps that follows an adopted one finds a stale tag
    a = _sim(cfg, B)
    monkeypatch.setenv('MATE_B200_REFILL', '0')
    b = _sim(cfg, B)
    a.reset(seed=21)
    b.reset(seed=21)
    stagger = np.random.RandomState(7).randint(0, 6, size=B).astype(np.int32)
    a.set_state({'episode_step': stagger})
    b.set_state({'episode_step': stagger})
    gen = torch.Generator(device='cuda')
    gen.manual_seed(4)
    scale = torch.tensor([cfg['camera_rotation_step'], cfg['camera_zooming_step']], device='cuda')
    for k in range(120):
        cam_act = (torch.rand((B, nc, 2), device='cuda', generator=gen) * 2 - 1) * scale
        tgt_act = (torch.rand((B, nt, 2), device='cuda', generator=gen) * 2 - 1) * cfg['target_step_size']
        (cam_a, tgt_a), rew_a, done_a = a.step(cam_act, tgt_act, auto_reset=True)   # no host synchronisation in between
        (cam_b, tgt_b), rew_b, done_b = b.step(cam_act, tgt_act, auto_reset=True)
        assert torch.equal(tgt_a, tgt_b) and torch.equal(cam_a, cam_b), k
        assert torch.equal(rew_a, rew_b) and torch.equal(done_a, done_b), k
    sa, sb = a.get_state(), b.get_state()
    for key in sa:
        assert (sa[key] == sb[key]).all(), key
    stats_a, stats_b = _np(a.episode_stats()), _np(b.episode_stats())
    assert stats_a[0] == stats_b[0] > B
    assert stats_a[6] + stats_a[7] == stats_a[0]
    assert stats_a[6] > 0 and stats_a[7] > 0, stats_a[:8]    # adopted AND computed in place
    assert stats_b[7] == stats_b[0]


def test_invalid_shape_and_alignment_errors():
    from mate_b200.config import flatten_config, read_config

    cfg = read_config('MATE-4v8-9.yaml')
    cfg['target']['location_random_range'] = cfg['target']['location_random_range'][:3]
    with pytest.raises(ValueError):
        _sim(flatten_config(cfg), 8)


@pytest.mark.parametrize('preset,overrides', [('MATE-4v8-9.yaml', {'max_episode_steps': 6}), ('MATE-Navigation.yaml', {'max_episode_steps': 5}),
                                              ('MATE-8v8-9.yaml', {'max_episode_steps': 6})])
def test_results_do_not_depend_on_the_warp_tile_size(preset, overrides, monkeypatch):
    """The step kernel cuts the batch into warp tiles of 32, 16 or 8 environments (chosen from the batch size,
    MATE_B200_TILE overrides it); draws are keyed on the global environment index, so every tile size gives the same
    bits -- including ragged last tiles, in-place resets and adopted prepared episodes."""
    from mate_b200.config import flatten_config, read_config

    cfg = flatten_config(read_config(preset, **overrides))
    nc, nt = cfg['num_cameras'], cfg['num_targets']
    B = 1003
    monkeypatch.setenv('MATE_B200_REFILL', '3')
    sims = []
    for tile in (32, 16, 8):
        monkeypatch.setenv('MATE_B200_TILE', str(tile))
        sims.append(_sim(cfg, B))
    first = [s.reset(seed=11) for s in sims]
    for other in first[1:]:
        assert torch.equal(first[0][1], other[1]) and (nc == 0 or torch.equal(first[0][0], other[0]))
    rng = np.random.RandomState(2)
    for k in range(20):
        cam_act = torch.from_numpy((rng.uniform(-1, 1, (B, nc, 2)) * [5.0, 2.5]).astype(np.float32)).cuda() if nc else None
        tgt_act = torch.from_numpy((rng.uniform(-1, 1, (B, nt, 2)) * 20.0).astype(np.float32)).cuda()
        outs = []
        for s in sims:
            (cam, tgt), rew, done = s.step(cam_act, tgt_act, auto_reset=True)
            outs.append((cam.clone() if nc else None, tgt.clone(), rew.clone(), done.clone()))
        for other in outs[1:]:
            assert torch.equal(outs[0][1], other[1]) and torch.equal(outs[0][2], other[2]) and torch.equal(outs[0][3], other[3]), k
            assert nc == 0 or torch.equal(outs[0][0], other[0]), k
    states = [s.get_state() for s in sims]
    for other in states[1:]:
        for key, value in states[0].items():
            assert np.array_equal(value, other[key]), key
    assert _np(sims[0].episode_stats())[0] >= 2 * B
