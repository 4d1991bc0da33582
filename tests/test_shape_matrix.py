"""Every compiled shape against an independent reference.

The library compiles one specialisation per (cameras, targets, obstacles) shape (``MATE_SHAPES`` in
``mate_b200/csrc/mate_b200.cu``), and the shape changes code paths, not only loop bounds: the row stores, the
obstacle rounds, the register arrays of the soft coverage and the lanes the greedy camera kernel gives one
environment.  ``SHAPES`` is the one list of them that the tests here iterate, and the first test keeps it equal to what
is compiled.  The GPU tests compare at every shape that has the entities they need:
- the soft coverage matrix (``BatchedSim.soft_coverage``) with the NumPy restatement ``oracle/soft_coverage_ref.py``, on
  states of the float64 C oracle and on a constructed batch of edge cases, and the auxiliary terms with
  ``test_aux_wrappers.terms_of``;
- the greedy camera and target kernels with ``oracle/greedy_camera_ref.py`` / ``greedy_target_ref.py`` in a closed loop
  through the oracle.
The step kernel itself is pinned to the oracle at every shape by ``test_cuda_parity.CASES``."""

import math
import os
import re
from fractions import Fraction

import numpy as np
import pytest

SHAPES = [(1, 1, 0), (1, 1, 9), (1, 2, 0), (1, 2, 9), (2, 2, 0), (2, 2, 9), (2, 4, 0), (2, 4, 9),
          (4, 2, 0), (4, 2, 9), (4, 4, 0), (4, 4, 9), (4, 8, 0), (4, 8, 9), (8, 8, 0), (8, 8, 9), (0, 8, 32)]
CAMERA_SHAPES = [s for s in SHAPES if s[0] > 0]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOFT_TOL = dict(rtol=2e-5, atol=2e-5)


def preset_of(shape):
    nc, nt, no = shape
    return 'MATE-Navigation.yaml' if nc == 0 else f'MATE-{nc}v{nt}-{no}.yaml'


def _ids(shapes):
    return [preset_of(s)[5:-5] for s in shapes]


def _flat(shape, **overrides):
    from mate_b200.config import flatten_config, read_config

    return flatten_config(read_config(preset_of(shape), **overrides))


def compiled_shapes(source):
    """The (cameras, targets, obstacles) list of the default branch of MATE_SHAPES in the text of mate_b200.cu."""
    match = re.search(r'#else\s*\n#define MATE_SHAPES\(X\)(.*?)#endif', source, re.S)
    assert match, 'the default branch of MATE_SHAPES was not found'
    return [tuple(int(v) for v in m) for m in re.findall(r'X\(\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*\)', match.group(1))]


# ---------------------------------------------------------------------------------------------------- the guard (CPU)
def test_matrix_equals_the_compiled_shapes():
    """SHAPES is what the library compiles, every shape is a preset of mate_b200.config and every preset one of the
    shapes (MATE.yaml is an alias of MATE-4v8-9.yaml), and the oracle parity cases of the step kernel cover them all."""
    from mate_b200.config import PRESETS, flatten_config, read_config

    with open(os.path.join(ROOT, 'mate_b200', 'csrc', 'mate_b200.cu'), encoding='utf-8') as f:
        compiled = compiled_shapes(f.read())
    assert len(set(compiled)) == len(compiled), compiled
    assert sorted(compiled) == sorted(SHAPES), (sorted(compiled), sorted(SHAPES))
    for shape in SHAPES:
        cfg = flatten_config(read_config(preset_of(shape)))
        assert (cfg['num_cameras'], cfg['num_targets'], cfg['num_obstacles']) == shape, shape
    assert PRESETS['MATE.yaml'] == PRESETS['MATE-4v8-9.yaml']
    assert sorted(set(PRESETS) - {'MATE.yaml'}) == sorted(preset_of(s) for s in SHAPES)
    import test_cuda_parity

    assert {case[0] for case in test_cuda_parity.CASES} == {preset_of(s) for s in SHAPES}


def test_the_guard_reads_every_line_of_the_shape_list():
    """compiled_shapes takes the default branch only, across its continuation lines; an added X(...) shows up."""
    text = ('#if defined(MATE_BASELINE_SHAPES)\n#define MATE_SHAPES(X) X(4, 2, 9)\n#else\n#define MATE_SHAPES(X)   \\\n'
            '    X(1, 1, 0) X(2, 2, 9)   \\\n    X(0, 8, 32)\n#endif\n')
    assert compiled_shapes(text) == [(1, 1, 0), (2, 2, 9), (0, 8, 32)]
    assert compiled_shapes(text.replace('X(0, 8, 32)', 'X(0, 8, 32) X(3, 3, 3)'))[-1] == (3, 3, 3)


# ----------------------------------------------------------------------------------------- the edge batch of the soft coverage
def _sectors(min_view):
    """(phi, theta) of the cameras of the edge batch: whole-degree left edges, edges at exactly -180 and +180, viewing
    angles of exactly 180 and of the minimum, sectors that straddle +-180 (camera c of environment e takes entry
    (e + c) % len)."""
    return [(-90.0, 180.0),                            # left edge -180, theta 180
            (90.0, 180.0),                             # right edge +180, theta 180
            (-180.0 + min_view / 2, min_view),         # left edge -180, minimum viewing angle
            (180.0 - min_view / 2, min_view),          # right edge +180, minimum viewing angle
            (-180.0, min_view),                        # straddles +-180
            (179.0, 180.0),                            # theta 180, straddles +-180 (left 89, right 269)
            (35.75, 47.5),                             # left edge 12 with a fractional width
            (-119.75, 60.5),                           # left edge -150
            (170.5, 61.0)]                             # left edge 140, straddles +-180


COLLAPSED_ENVS, NEAR_DISC_ENVS, NINE_DISC_ENVS = (0, 4), (1, 6), (2, 5)
SENSOR_TIE_ENVS = (9, 10, 11, 12)   # after the environments of the sectors


def _tie_decisions(ex, ey, thr):
    """(sqrt(ex^2 + ey^2) <= thr rounded term by term, {the same with either square fused into an FMA})."""
    def fused(a, b):   # fma(a, a, b * b): one rounding of the exact sum
        return float(Fraction(a) * Fraction(a) + Fraction(b * b))
    return math.sqrt(ex * ex + ey * ey) <= thr, {math.sqrt(fused(ex, ey)) <= thr, math.sqrt(fused(ey, ex)) <= thr}


def sensor_tie(anchor, thr):
    """A point at distance `thr` from `anchor` (float64 rounding) whose Sensor.perceive decision `distance <= thr` flips
    when the sum of squares is contracted into an FMA: a tie that only the reference's rounding decides."""
    for k in range(4000):
        a = 0.37 + 0.61 * k
        p = anchor + thr * np.array([np.cos(a), np.sin(a)])
        plain, fused = _tie_decisions(float(p[0] - anchor[0]), float(p[1] - anchor[1]), thr)
        if fused == {not plain}:
            return p
    raise AssertionError('no discriminating tie found')


def edge_states(cfg, seed=5):
    """A reset state of the oracle with every camera set to an edge sector and, per environment, target 0 or 1 exactly
    at camera 0 and the other on camera 0's arc of its sight range; with obstacles, camera 0 of COLLAPSED_ENVS inside a
    disc, a disc so close to camera 0 of NEAR_DISC_ENVS that its lattice has more than 120 rays, and every disc inside
    the sector of camera 0 of NINE_DISC_ENVS.  In SENSOR_TIE_ENVS, target 0 is a sensor_tie of camera 0 (target sight
    range + camera radius) and target 1 one of target 0 (target sight range)."""
    from oracle.oracle import Oracle

    nc, nt, no = cfg['num_cameras'], cfg['num_targets'], cfg['num_obstacles']
    min_view, rmax = cfg['camera_min_viewing_angle'], cfg['camera_max_sight_range']
    sectors = _sectors(min_view)
    B = len(sectors) + len(SENSOR_TIE_ENVS)
    ref = Oracle(cfg, B)
    ref.reset(seed=seed)
    st = ref.get_state()
    for e in range(B):
        for c in range(nc):
            st['cam_phi'][e, c], st['cam_theta'][e, c] = sectors[(e + c) % len(sectors)]
        phi0, theta0 = np.deg2rad(st['cam_phi'][e, 0]), st['cam_theta'][e, 0]
        cam0 = st['cam_xy'][e, 0].copy()
        if e in SENSOR_TIE_ENVS:
            st['tgt_xy'][e, 0] = sensor_tie(cam0, cfg['target_sight_range'] + cfg['camera_radius'])
            if nt > 1:
                st['tgt_xy'][e, 1] = sensor_tie(st['tgt_xy'][e, 0], cfg['target_sight_range'])
            continue
        if no and e in COLLAPSED_ENVS:
            cam0 = st['obs_xyr'][e, 0, :2] + [0.25 * st['obs_xyr'][e, 0, 2], 0.0]
            st['cam_xy'][e, 0] = cam0
        if no and e in NEAR_DISC_ENVS:   # r / d = 0.95: half opening angle 71.8 degrees, 143 lattice rays
            r = st['obs_xyr'][e, 0, 2]
            st['obs_xyr'][e, 0, :2] = cam0 + r / 0.95 * np.array([np.cos(phi0 + 0.2), np.sin(phi0 + 0.2)])
        if no and e in NINE_DISC_ENVS:
            d = rmax * (0.3 + 0.06 * np.arange(no))
            r = np.full(no, 25.0)
            spread = np.deg2rad(theta0 / 2 - np.rad2deg(np.arcsin(r / d)).max() - 0.5)
            bearing = phi0 + spread * (np.arange(no) - (no - 1) / 2) / ((no - 1) / 2)
            st['obs_xyr'][e, :, 0] = cam0[0] + d * np.cos(bearing)
            st['obs_xyr'][e, :, 1] = cam0[1] + d * np.sin(bearing)
            st['obs_xyr'][e, :, 2] = r
        at_camera, on_arc = e % 2, (e + 1) % 2
        st['tgt_xy'][e, at_camera % nt] = cam0
        if nt > 1:
            arc = np.sqrt(min_view * rmax * rmax / theta0)
            st['tgt_xy'][e, on_arc] = cam0 + arc * np.array([np.cos(phi0), np.sin(phi0)])
    ref.set_state(st)
    return ref.get_state()


@pytest.mark.parametrize('shape', CAMERA_SHAPES, ids=_ids(CAMERA_SHAPES))
def test_edge_batch_hits_its_edge_cases(shape):
    """CPU: the constructed batch survives the oracle's state round trip and really holds the edge cases the GPU test
    relies on, so that a later edit cannot quietly drop one."""
    from oracle import soft_coverage_ref as sr
    from oracle.oracle import Oracle

    cfg = _flat(shape)
    nc, nt, no = shape
    min_view, rmax = cfg['camera_min_viewing_angle'], cfg['camera_max_sight_range']
    st = edge_states(cfg)
    B = len(st['cam_phi'])
    assert B % 2 == 1 and B == len(_sectors(min_view)) + len(SENSOR_TIE_ENVS)
    ref = Oracle(cfg, B)
    ref.set_state(st)
    phi, theta = st['cam_phi'], st['cam_theta']
    left = sr.norm_angle(phi - theta / 2)
    assert (left == np.floor(left)).mean() > 0.7                           # sector edges on whole degrees
    assert (left == -180.0).any() and (left + theta == 180.0).any()        # left edge -180, right edge +180 exactly
    assert (theta == 180.0).any() and (theta == min_view).any()
    assert (left + theta > 180.0).any()                                    # sectors that wrap past +-180
    if nc >= 4:
        assert (left[theta == 180.0] == -180.0).any() and (left[theta == min_view] == -180.0).any()
    for e in SENSOR_TIE_ENVS:   # ties that rounding with an FMA would decide the other way
        pairs = [(st['tgt_xy'][e, 0], st['cam_xy'][e, 0], cfg['target_sight_range'] + cfg['camera_radius'])]
        if nt > 1:
            pairs.append((st['tgt_xy'][e, 1], st['tgt_xy'][e, 0], cfg['target_sight_range']))
        for p, q, thr in pairs:
            plain, fused = _tie_decisions(float(p[0] - q[0]), float(p[1] - q[1]), thr)
            assert fused == {not plain} and abs(np.hypot(*(p - q)) - thr) < 1e-9 * thr
    for e in range(len(_sectors(min_view))):
        cam0 = st['cam_xy'][e, 0]
        dist = np.hypot(*(st['tgt_xy'][e] - cam0).T)
        assert (dist == 0.0).any()                                         # a target exactly at the camera
        if nt > 1:
            arc = np.sqrt(min_view * rmax * rmax / theta[e, 0])
            assert np.isclose(dist, arc, rtol=1e-12, atol=0).any()         # and one on the arc
    if not no:
        return
    for e in COLLAPSED_ENVS:
        fov_phi, fov_rho = ref.get_fov(e, 0)
        assert len(fov_rho) and not fov_rho.any()                          # the collapsed boundary
        angles, norms, _ = sr.outer_samples(st['cam_xy'][e, 0], st['obs_xyr'][e], rmax)
        assert len(angles) == 4 and not norms.any()
    for e in NEAR_DISC_ENVS:
        rel = st['obs_xyr'][e, 0, :2] - st['cam_xy'][e, 0]
        half = np.rad2deg(np.arcsin(st['obs_xyr'][e, 0, 2] / np.hypot(*rel)))
        assert int(2 * half) > 120
        bearing = np.rad2deg(np.arctan2(rel[1], rel[0]))
        assert abs(sr.norm_angle(bearing - phi[e, 0])) < theta[e, 0] / 2    # and it faces the camera
    for e in NINE_DISC_ENVS:
        rel = st['obs_xyr'][e, :, :2] - st['cam_xy'][e, 0]
        d = np.hypot(rel[:, 0], rel[:, 1])
        half = np.rad2deg(np.arcsin(st['obs_xyr'][e, :, 2] / d))
        offset = np.abs(sr.norm_angle(np.rad2deg(np.arctan2(rel[:, 1], rel[:, 0])) - phi[e, 0]))
        assert (d + st['obs_xyr'][e, :, 2] < rmax).all() and (offset + half < theta[e, 0] / 2).all()


# ------------------------------------------------------------------------------------- soft coverage + auxiliary terms (GPU)
def _oracle_checkpoints(cfg, B, seed, limit, steps=(0, 11, 23)):
    """States of the oracle at the given step counts of an auto-resetting run (staggered episodes of `limit` steps,
    goal-seeking and random actions), with the rewards of the step that led there; and, for the first step after 4 whose
    auto-resets hit some but not all environments, (state before, actions, done)."""
    from oracle.oracle import Oracle
    from test_cuda_parity import _goal_seeking_actions

    nc, nt = cfg['num_cameras'], cfg['num_targets']
    ref = Oracle(cfg, B, num_threads=8)
    ref.reset(seed=seed)
    rng = np.random.RandomState(seed)
    st = ref.get_state()
    st['episode_step'] = rng.randint(0, limit, size=B).astype(np.int32)
    ref.set_state(st)
    out, reset_step = [], None
    rew = np.zeros((B, 2))
    for k in range(max(steps) + 1):
        if k in steps:
            out.append((ref.get_state(), rew))
        if k == max(steps):
            break
        before = ref.get_state()
        if k % 3 == 2:
            cam_act = (rng.uniform(-1, 1, (B, nc, 2)) * [cfg['camera_rotation_step'], cfg['camera_zooming_step']]).astype(np.float32)
            tgt_act = (rng.uniform(-1, 1, (B, nt, 2)) * cfg['target_step_size']).astype(np.float32)
        else:
            cam_act, tgt_act = _goal_seeking_actions(rng, cfg, before, B)
        _, rew, done = ref.step(cam_act, tgt_act, seed=seed, auto_reset=True)
        if reset_step is None and k > 4 and 0 < done.sum() < B:
            reset_step = (before, cam_act, tgt_act, done.copy())
    assert reset_step is not None
    return out, reset_step


def _empty_bits(bits):
    return (np.asarray(bits)[..., None].astype(np.int64) >> np.arange(4)) & 1


def _compare_soft_and_terms(cfg, states, rewards, transmit, ctx):
    """observe(aux=True) of `states` on both sides with the transmission draws replayed; mask_ct bit-exact, the kernel's
    soft coverage against the restatement (exactly tangent rays not cut), the auxiliary terms against terms_of.  Returns
    (entries, entries that match only the restatement that cuts exactly tangent rays)."""
    import torch

    from mate_b200.sim import BatchedSim
    from oracle import soft_coverage_ref as sr
    from oracle.oracle import Oracle
    from test_aux_wrappers import terms_of

    nc, nt = cfg['num_cameras'], cfg['num_targets']
    B = len(states['cam_phi'])
    rmax = cfg['camera_max_sight_range']
    area_product = cfg['camera_min_viewing_angle'] * rmax ** 2
    ref = Oracle(cfg, B, num_threads=8)
    ref.set_state(states)
    raux = ref.alloc_aux()
    ref.observe(transmit, aux=raux)
    sim = BatchedSim(cfg, B, device=0)
    sim.set_state(states)
    sim.observe(replay=(transmit, None), aux=True)
    for key in ('mask_ct', 'mask_cc', 'mask_co', 'mask_tc', 'mask_to', 'mask_tt', 'target_dones', 'is_colliding'):
        np.testing.assert_array_equal(sim.aux[key].cpu().numpy(), raux[key], err_msg=f'{ctx} {key}')
    for key in ('tgt_goal', 'tgt_empty_bits'):   # the oracle leaves these to its state
        np.testing.assert_array_equal(sim.aux[key].cpu().numpy(), states[key], err_msg=f'{ctx} {key}')
    np.testing.assert_allclose(sim.aux['coverage'].cpu().numpy(), raux['coverage'], rtol=1e-6, atol=1e-7, err_msg=ctx)
    got = sim.soft_coverage(auto_reset=False).cpu().numpy()
    sim.rewards.copy_(torch.from_numpy(rewards.astype(np.float32)))
    cam_terms, tgt_terms = (t.cpu().numpy() for t in sim.auxiliary_terms(sim.soft_coverage(auto_reset=False)))
    tangent = 0
    for b in range(B):
        tables = [ref.get_fov(b, c) for c in range(nc)]
        args = (states['cam_xy'][b], states['cam_phi'][b], states['cam_theta'][b], rmax, area_product, states['obs_xyr'][b],
                states['tgt_xy'][b], raux['mask_ct'][b].astype(bool), tables)
        want = sr.soft_coverage_matrix(*args, tangent_eps=1e-9)
        off = ~np.isclose(got[b], want, **SOFT_TOL)
        if off.any():   # only the documented tangent-ray class may differ: the restatement that cuts them must match
            cut = sr.soft_coverage_matrix(*args, tangent_eps=-1e-9)
            np.testing.assert_allclose(got[b][off], cut[off], **SOFT_TOL, err_msg=f'{ctx} env {b}: {np.argwhere(off)}')
            tangent += int(off.sum())
        cam, tgt = terms_of(nc, nt, rewards[b].astype(np.float32), raux['coverage'][b], raux['mask_ct'][b], raux['mask_tc'][b],
                            states['tgt_xy'][b], _empty_bits(states['tgt_empty_bits'][b]), states['tgt_goal'][b], raux['target_dones'][b],
                            raux['is_colliding'][b], soft=got[b])
        np.testing.assert_allclose(cam_terms[b], cam, rtol=1e-5, atol=1e-5, err_msg=f'{ctx} env {b} camera terms')
        np.testing.assert_allclose(tgt_terms[b], tgt, rtol=1e-5, atol=1e-5, err_msg=f'{ctx} env {b} target terms')
    sim.close()
    return got.size, tangent


@pytest.mark.gpu
@pytest.mark.parametrize('shape', CAMERA_SHAPES, ids=_ids(CAMERA_SHAPES))
def test_soft_coverage_and_terms_at_every_shape(shape):
    """GPU: the soft coverage kernels and the auxiliary terms kernel against their NumPy restatements on oracle states
    (after reset, mid-episode, after auto-resets; B odd, so the last block of (environment, camera) warps is partly
    empty at one and two cameras) and on the edge batch; soft_coverage(auto_reset=True) zeroes exactly the environments
    the last step reset."""
    import torch

    from mate_b200.sim import BatchedSim

    nc, nt, no = shape
    limit, seed, B = 23, 31, 37
    cfg = _flat(shape, max_episode_steps=limit)
    rng = np.random.RandomState(7)
    checkpoints, (before, cam_act, tgt_act, rdone) = _oracle_checkpoints(cfg, B, seed, limit)
    entries = tangent = 0
    for i, (states, rewards) in enumerate(checkpoints):
        n, k = _compare_soft_and_terms(cfg, states, rewards, rng.randint(0, 2, (B, nc, nt)).astype(np.uint8), f'{shape} checkpoint {i}')
        entries, tangent = entries + n, tangent + k
    edge = edge_states(cfg)
    n, k = _compare_soft_and_terms(cfg, edge, rng.uniform(-1, 1, (len(edge['cam_phi']), 2)), rng.randint(0, 2, (len(edge['cam_phi']), nc, nt)).astype(np.uint8),
                                   f'{shape} edge batch')
    entries, tangent = entries + n, tangent + k
    # measured on these states: no tangent-ray entry at any shape; the class may take a few, never without obstacles
    assert tangent <= 2 and (no or tangent == 0), (tangent, entries)

    # the auto-reset zeros, after a step whose time limit reset some environments
    sim = BatchedSim(cfg, B, device=0)
    sim.set_state(before)
    sim.step(torch.from_numpy(cam_act).cuda(), torch.from_numpy(tgt_act).cuda(), auto_reset=True, aux=True)
    done = sim.done.cpu().numpy().astype(bool)
    np.testing.assert_array_equal(done, rdone.astype(bool))
    zeroed = sim.soft_coverage(auto_reset=True).cpu().numpy().copy()
    plain = sim.soft_coverage(auto_reset=False).cpu().numpy()
    assert not zeroed[done].any()
    np.testing.assert_array_equal(zeroed[~done], plain[~done])
    assert plain[done].any()    # the reset environments do have a non-zero matrix of their own
    sim.close()


# ------------------------------------------------------------------------------------------- greedy agents, closed loop (GPU)
def _pack_camera(mem, nc, nt):
    return np.concatenate([mem['memory'].reshape(nc, 4 * nt), mem['time2forget'], mem['never_loaded'], mem['prev_action'],
                           mem['delay'], mem['neighbors'][:, None], mem['has_state'][:, None]], axis=-1).astype(np.float64)


def _pack_target(mem):
    return np.concatenate([mem['goal'][:, None], mem['non_empty'][:, None], mem['prev_xy'], mem['prev_noise']], axis=-1).astype(np.float64)


def _compare_memory(got, want, int_cols, ctx, loose_cols=()):
    """Agent memory: the integer fields exactly, the doubles to 1e-12 (`loose_cols`: previous actions, 1e-9)."""
    got, want = got.reshape(-1, got.shape[-1]), want.reshape(-1, want.shape[-1])
    cols = np.arange(got.shape[-1])
    exact = np.isin(cols, int_cols)
    loose = np.isin(cols, loose_cols)
    np.testing.assert_array_equal(got[:, exact], want[:, exact], err_msg=ctx)
    np.testing.assert_allclose(got[:, ~exact & ~loose], want[:, ~exact & ~loose], rtol=0, atol=1e-12, err_msg=ctx)
    np.testing.assert_allclose(got[:, loose], want[:, loose], rtol=0, atol=1e-9, err_msg=ctx)


@pytest.mark.gpu
@pytest.mark.parametrize('shape', SHAPES, ids=_ids(SHAPES))
def test_greedy_agents_at_every_shape(shape):
    """GPU: the greedy target and camera kernels against their restatements for 30 steps of a closed loop.  The oracle
    holds the state and steps with the restatement's actions (float32); every step the state is copied into a
    BatchedSim, the same seeded draws go to the kernels and to the restatements, and the cameras track the oracle's
    mask_ct.  The cameras of neighbouring environments stand far apart, and B * Nc is not a multiple of 32, so the camera kernel's
    last warp is partial.  Halfway through a random
    subset of environments is reset; its expected memory is the reset branch of the kernels (greedy.py:44-66 and
    265-277) followed by the restatement's step."""
    import torch

    import mate_b200
    from mate_b200.sim import BatchedSim
    from oracle.greedy_camera_ref import team_step as camera_step
    from oracle.greedy_target_ref import communicated_non_empty, team_step as target_step
    from oracle.oracle import Oracle

    nc, nt, no = shape
    B, steps, seed = 45, 30, 17
    cfg = _flat(shape)
    min_view, rmax = cfg['camera_min_viewing_angle'] if nc else 0.0, cfg['camera_max_sight_range'] if nc else 0.0
    rot, zoom = (cfg['camera_rotation_step'], cfg['camera_zooming_step']) if nc else (0.0, 0.0)
    ref = Oracle(cfg, B, num_threads=8)
    ref.reset(seed=seed)
    if nc:   # the presets put the cameras of every environment at the same places (at 1 and 2 cameras fixed ones): here the
        # cameras of environment e stand within 150 of warehouse e % 4, so that the camera kernel's lanes of neighbouring
        # environments hold locations 1850 apart
        st = ref.get_state()
        pos = np.random.RandomState(seed)
        corner = 800.0 * np.array([[1.0, 1.0], [-1.0, 1.0], [-1.0, -1.0], [1.0, -1.0]])[np.arange(B) % 4]
        st['cam_xy'] = corner[:, None, :] + pos.uniform(-150.0, 150.0, st['cam_xy'].shape)
        ref.set_state(st)
    raux = ref.alloc_aux()
    ref.observe(aux=raux)
    sim = BatchedSim(cfg, B, device=0)
    targets = mate_b200.GreedyTargetAgent(seed=1)
    targets.bind(sim)
    if nc:
        cameras = mate_b200.GreedyCameraAgent(seed=2)
        cameras.bind(sim)
    rng = np.random.default_rng(seed)
    st = ref.get_state()
    tmem = [{'goal': np.full(nt, -1, dtype=np.int64), 'non_empty': np.full(nt, 15, dtype=np.int64), 'prev_xy': st['tgt_xy'][b].copy(),
             'prev_noise': np.zeros((nt, 2))} for b in range(B)]
    cmem = [{'memory': np.zeros((nc, nt, 4)), 'time2forget': np.zeros((nc, nt)), 'never_loaded': np.ones((nc, nt)),
             'prev_action': np.zeros((nc, 2)), 'delay': np.zeros((nc, nc)), 'neighbors': np.zeros(nc, dtype=np.int64),
             'has_state': np.ones(nc, dtype=np.int64)} for b in range(B)]
    targets.memory.copy_(torch.from_numpy(np.stack([_pack_target(m) for m in tmem])))
    if nc:
        cameras.memory.copy_(torch.from_numpy(np.stack([_pack_camera(m, nc, nt) for m in cmem])))
    resets = tracked = 0
    for k in range(steps):
        ctx = f'{shape} step {k}'
        st = ref.get_state()
        sim.set_state(st)
        mask_ct = raux['mask_ct'].astype(bool)
        tracked += int(mask_ct.sum())
        reset = rng.random(B) < 0.4 if k == steps // 2 else np.zeros(B, dtype=bool)
        resets += int(reset.sum())
        step_size = cfg['target_step_size'] / st['tgt_capacity']
        empty = _empty_bits(st['tgt_empty_bits']).astype(bool)
        has_goal = (st['tgt_goal'] >= 0) & (st['tgt_weight'] > 0)
        # target draws; reset(observation): goal from the state, every warehouse non-empty, previous location = location,
        # previous noise = half of a uniform sample (mate_agents.cuh greedy_target_kernel, greedy.py:265-277)
        t_draws = {'binomial': rng.integers(0, 2, (B, nt)).astype(np.uint8), 'sample': rng.uniform(-1, 1, (B, nt, 2)) * step_size[..., None],
                   'reset_sample': rng.uniform(-1, 1, (B, nt, 2)) * step_size[..., None], 'choice': np.full((B, nt), -1, dtype=np.int8)}
        for b in np.flatnonzero(reset):
            tmem[b] = {'goal': np.where(has_goal[b], st['tgt_goal'][b], -1).astype(np.int64), 'non_empty': np.full(nt, 15, dtype=np.int64),
                       'prev_xy': st['tgt_xy'][b].copy(), 'prev_noise': 0.5 * t_draws['reset_sample'][b]}
        for b in range(B):   # the goal choice: a member of the set the agent holds after communicating
            non_empty = communicated_non_empty(empty[b], tmem[b]['non_empty'])
            for t in range(nt):
                if non_empty[t]:
                    t_draws['choice'][b, t] = rng.choice(np.flatnonzero((non_empty[t] >> np.arange(4)) & 1))
        goal_bits = np.zeros((B, nt, 4))
        for b, t in zip(*np.nonzero(st['tgt_goal'] >= 0)):
            goal_bits[b, t, st['tgt_goal'][b, t]] = st['tgt_weight'][b, t]
        tgt_act = np.zeros((B, nt, 2))
        for b in range(B):
            tgt_act[b], tmem[b] = target_step(st['tgt_xy'][b], step_size[b], goal_bits[b], empty[b], tmem[b],
                                              {n: t_draws[n][b] for n in ('binomial', 'sample', 'choice')}, targets.noise_scale)
        got = targets.act(reset_mask=torch.from_numpy(reset.astype(np.uint8)).cuda(), replay=t_draws).cpu().numpy()
        np.testing.assert_allclose(got, tgt_act, rtol=1e-6, atol=1e-5, err_msg=ctx)
        _compare_memory(targets.memory.cpu().numpy(), np.stack([_pack_target(m) for m in tmem]), [0, 1], ctx + ' target memory')
        cam_act = np.zeros((B, nc, 2))
        if nc:
            # camera draws; reset(observation): tracked targets remembered, untracked ones zero, every target never loaded,
            # no delays, no known teammates, the own state still to send (mate_agents.cuh greedy_camera_kernel, greedy.py:44-66)
            c_draws = {'binomial': rng.integers(0, 2, (B, nc)).astype(np.int8),
                       'sample': rng.uniform(-1, 1, (B, nc, 2)) * [rot, zoom], 'delay': rng.integers(6, 50, (B, nc, nc)).astype(np.int32)}
            loaded = has_goal.astype(float)
            tgt_state = np.concatenate([st['tgt_xy'], np.full((B, nt, 1), cfg['target_sight_range']), loaded[..., None]], axis=-1)
            for b in np.flatnonzero(reset):
                seen = mask_ct[b]
                cmem[b] = {'memory': np.where(seen[..., None], tgt_state[b][None], 0.0), 'time2forget': np.where(seen, 25.0, 0.0),
                           'never_loaded': np.ones((nc, nt)), 'prev_action': np.zeros((nc, 2)), 'delay': np.zeros((nc, nc)),
                           'neighbors': np.zeros(nc, dtype=np.int64), 'has_state': np.ones(nc, dtype=np.int64)}
            for b in range(B):
                cam_act[b], cmem[b] = camera_step(st['cam_xy'][b], st['cam_phi'][b], st['cam_theta'][b], tgt_state[b], mask_ct[b], cmem[b],
                                                  {n: c_draws[n][b] for n in c_draws}, (min_view, rmax, rot, zoom))
            got = cameras.act(raux['mask_ct'], reset_mask=torch.from_numpy(reset.astype(np.uint8)).cuda(), replay=c_draws).cpu().numpy()
            np.testing.assert_allclose(got, cam_act, rtol=1e-6, atol=1e-5, err_msg=ctx)
            ints = list(range(4 * nt, 6 * nt)) + list(range(6 * nt + 2, 6 * nt + 4 + nc))   # time2forget, never_loaded, delays, bit sets
            _compare_memory(cameras.memory.cpu().numpy(), np.stack([_pack_camera(m, nc, nt) for m in cmem]), ints, ctx + ' camera memory',
                            loose_cols=[6 * nt, 6 * nt + 1])
        ref.step(cam_act.astype(np.float32), tgt_act.astype(np.float32), seed=seed, auto_reset=False, aux=raux)
    assert resets > 0 and (tracked > 0 or nc == 0)
    sim.close()
