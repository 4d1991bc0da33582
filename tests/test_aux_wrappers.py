"""Auxiliary-reward / training-information wrappers (SURVEY.md section 8f, N3) against the reference's own wrapper
classes: ``tests/golden/aux_*.npz`` hold, for sampled steps of greedy-agent episodes, the state before the step, the
action, the recorded draws, and what ``MoreTrainingInformation`` / ``AuxiliaryCameraRewards`` /
``AuxiliaryTargetRewards`` of the reference reported after it (written by ``oracle/gen_aux_golden.py``)."""

import glob
import os

import numpy as np
import pytest

import golden_util as gu

NAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(gu.GOLDEN_DIR, 'aux_*.npz')))
WAREHOUSES = np.array([[925.0, 925.0], [-925.0, 925.0], [-925.0, -925.0], [925.0, -925.0]])   # constants.py:70-72
CAM_SOFT, TGT_SOFT = 4, 6   # column of soft_coverage_score in the two key lists


def terms_numpy(g, i):
    """Plain restatement of the terms (auxiliary_camera_rewards.py:140-149, auxiliary_target_rewards.py:135-177,
    more_training_information.py:61-82) from the recorded after-step pieces of sample i."""
    nc, nt, _ = (int(x) for x in g['cfg_counts'])
    return terms_of(nc, nt, g['a_out_team_reward'][i], g['a_out_tgt_terms'][i][0, 1:4], g['a_out_mask_ct'][i], g['a_out_mask_tc'][i],
                    g['a_out_tgt_xy'][i], g['a_out_tgt_empty_bits'][i], g['a_out_tgt_goal'][i], g['a_out_tgt_individual_done'][i],
                    g['a_out_tgt_is_colliding'][i])


def terms_of(nc, nt, team_reward, cov, mask_ct, mask_tc, xy, empty, goal, individual_done, is_colliding, soft=None):
    """The terms of one environment: ``team_reward`` [2], ``cov`` the three coverage rates, masks [Nc, Nt] / [Nt, Nc],
    target locations [Nt, 2], empty bits [Nt, 4], goals, individual done and collision flags [Nt]; ``soft`` [Nc, Nt]
    (``None``: the soft_coverage_score columns stay 0) aggregated like auxiliary_camera_rewards.py:130-138 and
    auxiliary_target_rewards.py:151-162."""
    mask_ct, mask_tc = np.asarray(mask_ct).astype(bool), np.asarray(mask_tc).astype(bool)
    cam_soft, tgt_soft = np.zeros(nc), np.zeros(nt)
    if soft is not None and nc:
        soft = np.asarray(soft, dtype=np.float64)
        cam_soft = np.where(mask_ct.any(-1), (soft * mask_ct).sum(-1), np.tanh(soft.max(-1)))
        tgt_soft = np.where(mask_ct.any(-2), (soft * mask_ct).sum(-2), np.tanh(soft.max(-2)))
    cam = np.zeros((nc, 8))
    for c in range(nc):
        cam[c] = [team_reward[0], cov[0], cov[1], cov[2], cam_soft[c], mask_ct[c].sum(), 1.0, mask_tc[:, c].any()]
    tgt = np.zeros((nt, 16))
    empty = np.asarray(empty).astype(bool)
    for t in range(nt):
        wd = np.maximum(np.linalg.norm(xy[t] - WAREHOUSES, axis=-1) - 75.0, 0.0)
        if goal[t] >= 0:
            goal_distance = wd[goal[t]]
        elif not empty[t].all():
            goal_distance = wd[~empty[t]].min()
        else:
            goal_distance = 1000.0
        tgt[t, :10] = [team_reward[1], cov[0], cov[1], cov[2], goal_distance / 2000.0, individual_done[t],
                       tgt_soft[t], mask_ct[:, t].any() if nc else 0.0, is_colliding[t], 1.0]
        tgt[t, 10] = goal[t]
        tgt[t, 11] = wd[goal[t]] if goal[t] >= 0 else 1000.0
        tgt[t, 12:16] = wd
    return cam, tgt


def expected(g):
    """Golden terms with the soft coverage score (not built) zeroed, and the rewards without its contribution."""
    cam_terms, tgt_terms = g['a_out_cam_terms'].copy(), g['a_out_tgt_terms'].copy()
    nc = int(g['cfg_counts'][0])
    cam_reward = g['a_out_cam_reward'] - g['camera_coef'][CAM_SOFT] * cam_terms[..., CAM_SOFT] if nc else g['a_out_cam_reward']
    tgt_reward = g['a_out_tgt_reward'] - g['target_coef'][TGT_SOFT] * tgt_terms[..., TGT_SOFT]
    cam_terms[..., CAM_SOFT] = 0.0
    tgt_terms[..., TGT_SOFT] = 0.0
    return cam_terms, tgt_terms, cam_reward, tgt_reward


@pytest.mark.parametrize('name', NAMES)
def test_term_formulas_match_the_reference_wrappers(name):
    """CPU: the formulas the CUDA kernel implements reproduce the reference wrappers' info entries."""
    g = gu.load(name)
    cam_terms, tgt_terms, _, _ = expected(g)
    for i in range(int(g['count'])):
        cam, tgt = terms_numpy(g, i)
        np.testing.assert_allclose(cam[:, :7], cam_terms[i], rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(tgt[:, :10], tgt_terms[i], rtol=1e-12, atol=1e-12)
        np.testing.assert_array_equal(cam[:, 5], g['a_out_cam_num_tracked'][i])
        np.testing.assert_array_equal(cam[:, 7], g['a_out_cam_is_sensed'][i])
        np.testing.assert_allclose(tgt[:, 11], g['a_out_tgt_goal_distance'][i], rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(tgt[:, 12:16], g['a_out_tgt_warehouse_distances'][i], rtol=1e-12, atol=1e-12)
        np.testing.assert_array_equal(tgt[:, 7], g['a_out_tgt_is_tracked'][i])


def test_wrapper_assertions():
    """Ordering / key rules of the reference (auxiliary_camera_rewards.py:60-82)."""
    from mate_b200 import wrappers

    class Fake:
        num_cameras = 4
        unwrapped = None

    fake = Fake()
    fake.unwrapped = fake
    inner = wrappers.Wrapper(fake)
    with pytest.raises(AssertionError):
        wrappers.AuxiliaryCameraRewards(inner, coefficients={'raw_reward': 1.0})   # needs RepeatedRewardIndividualDone
    repeated = wrappers.RepeatedRewardIndividualDone(inner)
    with pytest.raises(AssertionError):
        wrappers.AuxiliaryCameraRewards(repeated, coefficients={'no_such_key': 1.0})
    with pytest.raises(AssertionError):
        wrappers.AuxiliaryTargetRewards(repeated, coefficients={'raw_reward': 1.0}, reduction='median')
    once = wrappers.AuxiliaryTargetRewards(repeated, coefficients={'raw_reward': 1.0})
    with pytest.raises(AssertionError):
        wrappers.AuxiliaryTargetRewards(once, coefficients={'raw_reward': 1.0})


@pytest.mark.gpu
@pytest.mark.parametrize('name', NAMES)
def test_auxiliary_wrappers_match_the_reference(name):
    """GPU: every sampled reference state is injected into its own environment of one batch, the recorded step is
    repeated (recorded action and draws), and the wrapper stack's rewards and infos are compared with the
    reference's."""
    import torch

    import mate_b200

    g = gu.load(name)
    nc, nt, _ = (int(x) for x in g['cfg_counts'])
    count = int(g['count'])
    config = str(g['config_name'])
    cam_keys, tgt_keys = [str(k) for k in g['camera_keys']], [str(k) for k in g['target_keys']]
    cam_coef = {k: float(v) for k, v in zip(cam_keys, g['camera_coef']) if k != 'soft_coverage_score'}
    tgt_coef = {k: float(v) for k, v in zip(tgt_keys, g['target_coef']) if k != 'soft_coverage_score'}
    wrappers = [mate_b200.MoreTrainingInformation, mate_b200.RepeatedRewardIndividualDone]
    if nc:
        wrappers.append(lambda env: mate_b200.AuxiliaryCameraRewards(env, coefficients=cam_coef))
    wrappers.append(lambda env: mate_b200.AuxiliaryTargetRewards(env, coefficients=tgt_coef))
    env = mate_b200.make('MultiAgentTracking-v0', config=config, num_envs=count, wrappers=wrappers)
    base = env.unwrapped
    base.set_state(gu.stack_states([gu.state_arrays(g, 'a_', i) for i in range(count)]))
    base.replay_next = (g['a_transmit'], g['a_goal_choice'])
    cam_act = torch.from_numpy(g['a_cam_act'].astype(np.float32)).cuda()
    tgt_act = torch.from_numpy(g['a_tgt_act'].astype(np.float32)).cuda()
    _, (cam_reward, tgt_reward), _, (cam_infos, tgt_infos) = env.step((cam_act, tgt_act))
    torch.cuda.synchronize()
    exp_cam_terms, exp_tgt_terms, exp_cam_reward, exp_tgt_reward = expected(g)
    cam_terms, tgt_terms = (t.cpu().numpy() for t in base.auxiliary_terms())
    # the step itself must have reproduced the reference (masks bit-exact), otherwise the comparison is void
    np.testing.assert_array_equal(base.camera_target_view_mask.cpu().numpy(), g['a_out_mask_ct'].astype(bool))
    np.testing.assert_array_equal(base.target_camera_view_mask.cpu().numpy(), g['a_out_mask_tc'].astype(bool))
    tol = dict(rtol=1e-5, atol=1e-5)
    if nc:
        np.testing.assert_allclose(cam_terms[..., :7], exp_cam_terms, **tol)
        np.testing.assert_allclose(cam_reward.cpu().numpy(), exp_cam_reward, rtol=1e-5, atol=1e-3)
        np.testing.assert_array_equal(cam_infos['num_tracked'].cpu().numpy(), g['a_out_cam_num_tracked'])
        np.testing.assert_array_equal(cam_infos['is_sensed'].cpu().numpy(), g['a_out_cam_is_sensed'].astype(bool))
        np.testing.assert_allclose(cam_infos['auxiliary_reward_coverage_rate'].cpu().numpy(), exp_cam_terms[..., 1], **tol)
    np.testing.assert_allclose(tgt_terms[..., :10], exp_tgt_terms, **tol)
    np.testing.assert_allclose(tgt_reward.cpu().numpy(), exp_tgt_reward, rtol=1e-5, atol=1e-3)
    np.testing.assert_array_equal(tgt_infos['goal'].cpu().numpy(), g['a_out_tgt_goal'])
    # distances: float32 of a float64 norm minus the warehouse radius
    np.testing.assert_allclose(tgt_infos['goal_distance'].cpu().numpy(), g['a_out_tgt_goal_distance'], rtol=1e-5, atol=2e-4)
    np.testing.assert_allclose(tgt_infos['warehouse_distances'].cpu().numpy(), g['a_out_tgt_warehouse_distances'], rtol=1e-5, atol=2e-4)
    np.testing.assert_array_equal(tgt_infos['individual_done'].cpu().numpy(), g['a_out_tgt_individual_done'].astype(bool))
    np.testing.assert_array_equal(tgt_infos['is_tracked'].cpu().numpy(), g['a_out_tgt_is_tracked'].astype(bool))
    np.testing.assert_array_equal(tgt_infos['is_colliding'].cpu().numpy(), g['a_out_tgt_is_colliding'].astype(bool))
    np.testing.assert_allclose(tgt_infos['auxiliary_reward_normalized_goal_distance'].cpu().numpy(), exp_tgt_terms[..., 4], **tol)
    base.close()


def _soft_reference(g, limit):
    """(matrix without tangent cuts, matrix with tangent cuts) of the NumPy restatement for the first samples."""
    from oracle import soft_coverage_ref as sr
    from oracle.oracle import Oracle

    cfg = gu.flat_config(g)
    nc, rmax = cfg['num_cameras'], cfg['camera_max_sight_range']
    area_product = cfg['camera_min_viewing_angle'] * rmax ** 2
    sim = Oracle(cfg, 1)
    sim.set_state(gu.state_arrays(g, 'a_', 0))   # one episode per fixture: the geometry is that of sample 0
    tables = [sim.get_fov(0, c) for c in range(nc)]
    n = min(int(g['count']), limit)
    out = []
    for eps in (1e-9, -1e-9):
        rows = []
        for i in range(n):
            phi, theta = sr.after_step_cameras(g, i)
            rows.append(sr.soft_coverage_matrix(g['a_cam_xy'][i], phi, theta, rmax, area_product, g['a_obs_xyr'][i], g['a_out_tgt_xy'][i],
                                                g['a_out_mask_ct'][i].astype(bool), tables, tangent_eps=eps))
        out.append(np.array(rows))
    return out


@pytest.mark.parametrize('name', [n for n in NAMES if 'Navigation' not in n])
def test_soft_coverage_restatement_matches_the_reference(name):
    """CPU: the NumPy restatement of compute_soft_coverage_scores (the checker of the CUDA kernel) against ALL of the
    reference's recorded matrices.  The reference decides every exactly tangent boundary ray by rounding noise
    (DESIGN.md "Tangent rays"), independently per ray, so a recorded entry need not equal the restatement under one
    global convention; what is proven instead, entry by entry (``soft_coverage_explained``): the recorded value is the
    distance to a boundary point that SOME outcome of the tangent rays contains, and no point that every outcome
    contains is closer.  The share of entries that equal the convention of the CUDA path (no tangent ray cut) is
    reported and bounded."""
    from oracle import soft_coverage_ref as sr
    from oracle.oracle import Oracle

    g = gu.load(name)
    cfg = gu.flat_config(g)
    nc, rmax = cfg['num_cameras'], cfg['camera_max_sight_range']
    area_product = cfg['camera_min_viewing_angle'] * rmax ** 2
    sim = Oracle(cfg, 1)
    sim.set_state(gu.state_arrays(g, 'a_', 0))   # one episode per fixture: the geometry is that of sample 0
    tables = [sim.get_fov(0, c) for c in range(nc)]
    n = int(g['count'])
    same = total = 0
    unexplained = []
    for i in range(n):
        phi, theta = sr.after_step_cameras(g, i)
        ok, eq = sr.soft_coverage_explained(g['a_cam_xy'][i], phi, theta, rmax, area_product, g['a_obs_xyr'][i], g['a_out_tgt_xy'][i],
                                            g['a_out_mask_ct'][i].astype(bool), tables, g['a_out_soft_matrix'][i])
        same += int(eq.sum())
        total += ok.size
        for c, t in np.argwhere(~ok):
            plain = sr.soft_coverage_matrix(g['a_cam_xy'][i], phi, theta, rmax, area_product, g['a_obs_xyr'][i], g['a_out_tgt_xy'][i],
                                            g['a_out_mask_ct'][i].astype(bool), tables)[c, t]
            unexplained.append((i, int(c), int(t), float(theta[c]), float(abs(plain - g['a_out_soft_matrix'][i][c, t]))))
    # 40 383 of the 40 384 recorded entries are proven.  The one that is not (aux_4v8-9 sample 541, camera 3 at a
    # viewing angle of exactly 180 degrees, target 3) differs by 7.7e-4 at a value of 4.07 under every outcome of the
    # tangent rays; its cause is not identified.  More than that, or a larger deviation, fails.
    assert len(unexplained) <= 1 and all(dev < 1e-3 and theta == 180.0 for *_, theta, dev in unexplained), unexplained
    assert same / total > 0.85, same / total     # measured: 0.91 (4v8-9), 0.985 (8v8-9), 1.0 without obstacles
    if int(g['cfg_counts'][2]) == 0:
        assert same == total


@pytest.mark.gpu
@pytest.mark.parametrize('name', [n for n in NAMES if 'Navigation' not in n])
def test_soft_coverage_matches_the_restatement(name):
    """GPU: the soft coverage matrix of the recorded steps against the NumPy restatement (exactly tangent rays not
    cut, the convention of the CUDA path), and the soft_coverage_score terms of both teams against the reference's
    aggregation of it."""
    import torch

    import mate_b200

    g = gu.load(name)
    nc, nt, _ = (int(x) for x in g['cfg_counts'])
    limit = 256
    want, _ = _soft_reference(g, limit)
    n = len(want)
    env = mate_b200.make('MultiAgentTracking-v0', config=str(g['config_name']), num_envs=n, wrappers=[
        mate_b200.RepeatedRewardIndividualDone,
        lambda e: mate_b200.AuxiliaryCameraRewards(e, coefficients={'soft_coverage_score': 1.0}),
        lambda e: mate_b200.AuxiliaryTargetRewards(e, coefficients={'soft_coverage_score': 1.0})])
    base = env.unwrapped
    base.set_state(gu.stack_states([gu.state_arrays(g, 'a_', i) for i in range(n)]))
    base.replay_next = (g['a_transmit'][:n], g['a_goal_choice'][:n])
    cam_act = torch.from_numpy(g['a_cam_act'][:n].astype(np.float32)).cuda()
    tgt_act = torch.from_numpy(g['a_tgt_act'][:n].astype(np.float32)).cuda()
    _, (cam_reward, tgt_reward), (cam_done, _), _ = env.step((cam_act, tgt_act))
    torch.cuda.synchronize()
    live = ~cam_done[:, 0].cpu().numpy().astype(bool)     # auto-reset environments report zeros
    assert live.sum() >= n - 1
    mask = g['a_out_mask_ct'][:n].astype(bool)
    np.testing.assert_array_equal(base.camera_target_view_mask.cpu().numpy(), mask)
    got = base.sim._soft.cpu().numpy()  # pylint: disable=protected-access
    np.testing.assert_allclose(got[live], want[live], rtol=2e-5, atol=2e-5)
    # aggregation (auxiliary_camera_rewards.py:130-138, auxiliary_target_rewards.py:151-162)
    cam_want = np.where(mask.any(-1), (want * mask).sum(-1), np.tanh(want.max(-1)))
    tgt_want = np.where(mask.any(-2), (want * mask).sum(-2), np.tanh(want.max(-2)))
    np.testing.assert_allclose(cam_reward.cpu().numpy()[live], cam_want[live], rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(tgt_reward.cpu().numpy()[live], tgt_want[live], rtol=1e-4, atol=1e-4)
    assert not got[~live].any()
    base.close()


@pytest.mark.gpu
def test_reductions_and_callable_coefficients():
    """`reduction` shares one reward per team; a callable coefficient is called once per key with tensors."""
    import torch

    import mate_b200

    B = 32
    calls = []

    def schedule(agent_ids, episode_id, episode_step, raw_reward, value):
        calls.append((tuple(agent_ids.shape), episode_id, tuple(episode_step.shape), tuple(value.shape)))
        return 0.5 + 0.0 * value

    env = mate_b200.make('MultiAgentTracking-v0', config='MATE-4v8-9.yaml', num_envs=B, wrappers=[
        mate_b200.RepeatedRewardIndividualDone,
        lambda e: mate_b200.AuxiliaryCameraRewards(e, coefficients={'num_tracked': schedule, 'baseline': 2}, reduction='mean'),
        lambda e: mate_b200.AuxiliaryTargetRewards(e, coefficients={'raw_reward': 1.0, 'is_tracked': -1.0}, reduction='min')])
    env.reset(seed=11)
    rng = np.random.RandomState(1)
    cam_act = torch.from_numpy((rng.uniform(-1, 1, (B, 4, 2)) * [5.0, 2.5]).astype(np.float32)).cuda()
    tgt_act = torch.from_numpy((rng.uniform(-1, 1, (B, 8, 2)) * 20.0).astype(np.float32)).cuda()
    _, (cam_reward, tgt_reward), _, (cam_infos, tgt_infos) = env.step((cam_act, tgt_act))
    assert calls == [((1, 4), 0, (B, 1), (B, 4))]
    individual = 0.5 * cam_infos['auxiliary_reward_num_tracked'] + 2.0
    assert torch.allclose(cam_infos['reward'], individual)
    assert torch.allclose(cam_reward, individual.mean(dim=-1, keepdim=True).expand(-1, 4))
    assert torch.equal(cam_infos['shared_reward'], cam_reward)
    individual = tgt_infos['auxiliary_reward_raw_reward'] - tgt_infos['auxiliary_reward_is_tracked']
    assert torch.allclose(tgt_reward, individual.min(dim=-1, keepdim=True).values.expand(-1, 8))
    env.unwrapped.close()


@pytest.mark.gpu
def test_reference_compatible_single_env_types():
    """num_envs=None: the wrappers return the reference's types (lists of Python floats, list-of-dict infos)."""
    import mate_b200

    coefficients = {'raw_reward': 1.0, 'coverage_rate': 2.0, 'soft_coverage_score': 0.5, 'num_tracked': lambda c, ep, step, raw, value: 0.25}
    env = mate_b200.make('MultiAgentTracking-v0', config='MATE-4v2-9.yaml', wrappers=[
        mate_b200.MoreTrainingInformation, mate_b200.RepeatedRewardIndividualDone,
        lambda e: mate_b200.AuxiliaryCameraRewards(e, coefficients=coefficients, reduction='mean'),
        lambda e: mate_b200.AuxiliaryTargetRewards(e, coefficients={'normalized_goal_distance': -1.0, 'sparse_delivery': 10.0})])
    cam_obs, tgt_obs = env.reset(seed=2)
    assert isinstance(cam_obs, np.ndarray) and cam_obs.shape == (4, 96) and tgt_obs.shape == (2, 101)
    rng = np.random.RandomState(0)
    for _ in range(5):
        action = (rng.uniform(-1, 1, (4, 2)) * [5.0, 2.5], rng.uniform(-1, 1, (2, 2)) * 20.0)
        (cam_obs, tgt_obs), (cam_reward, tgt_reward), (cam_done, tgt_done), (cam_infos, tgt_infos) = env.step(action)
    assert isinstance(cam_reward, list) and len(cam_reward) == 4 and isinstance(cam_reward[0], float)
    assert isinstance(tgt_reward, list) and len(tgt_reward) == 2 and cam_done == [False] * 4 and tgt_done == [False] * 2
    assert len(cam_infos) == 4 and len(tgt_infos) == 2
    info = cam_infos[1]
    for key in ('num_tracked', 'is_sensed', 'auxiliary_reward_soft_coverage_score', 'reward_coefficient_num_tracked', 'reward',
                'shared_reward', 'camera_states', 'target_states', 'state', 'remaining_cargoes', 'camera_target_view_mask'):
        assert key in info, key
    assert info['reward_coefficient_num_tracked'] == 0.25 and cam_reward[0] == cam_reward[3] == info['shared_reward']
    expected = (info['auxiliary_reward_raw_reward'] + 2.0 * info['auxiliary_reward_coverage_rate']
                + 0.5 * info['auxiliary_reward_soft_coverage_score'] + 0.25 * info['auxiliary_reward_num_tracked'])
    assert abs(info['reward'] - expected) < 1e-4
    tinfo = tgt_infos[0]
    assert tinfo['goal'] in (-1, 0, 1, 2, 3) and len(tinfo['warehouse_distances']) == 4
    assert abs(tinfo['reward'] - (-tinfo['auxiliary_reward_normalized_goal_distance'] + 10.0 * tinfo['auxiliary_reward_sparse_delivery'])) < 1e-5
    assert info['state'].shape == env.unwrapped.state_space.shape
    env.unwrapped.close()
