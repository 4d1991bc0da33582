"""Communication wrappers (``RestrictedCommunicationRange``, ``RandomMessageDropout``, ``NoCommunication``; DESIGN.md
section 7h) for the batched greedy teams and for the host ``Message`` traffic of the single-environment mode.

The kernels are checked against the NumPy restatements ``oracle/greedy_*_ref.py`` (pinned to recorded reference agents
by ``tests/test_agents.py``) on the recorded states of ``tests/golden/agents_*.npz``: the filters only remove messages
from the restatements' receive phase, so the kernels' delivered bits fed into the restatements must reproduce the
kernels' memory and actions.  The filtered restatements below are built on the unmodified ``oracle`` functions: they
only take messages out of the receive phase."""

import os

import numpy as np
import pytest

import golden_util as gu
from oracle import greedy_camera_ref as camera_ref
from oracle import greedy_target_ref as target_ref

torch = pytest.importorskip('torch')

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, 'golden')
AGENT_NAMES = ['agents_4v8-9', 'agents_4v2-0']
NEAR_TIE = 1e-9


# ---------------------------------------------------------------------------------------------------------------------
# the restatements with communication wrappers: delivered [N, N] bool (default: all true), entry (s, r) = the message
# of s reaches r.  Each also reports 'sent' [N, N]: the messages of the step before any filter.
# ---------------------------------------------------------------------------------------------------------------------
def delivered_in_range(xy, range_limit):
    """RestrictedCommunicationRange on a state: entry (s, r) = agents s and r are at most ``range_limit`` apart, in the
    fp64 expression of the kernels (no fused multiply-add)."""
    xy = np.asarray(xy, dtype=np.float64)
    dx = xy[:, None, 0] - xy[None, :, 0]
    dy = xy[:, None, 1] - xy[None, :, 1]
    return np.sqrt(dx * dx + dy * dy) <= range_limit


def target_team_step(xy, step_size, goal_bits, empty_bits, memory, draws, noise_scale, delivered=None):
    """``oracle.greedy_target_ref.team_step`` with filtered broadcasts.  process_messages (greedy.py:330-336) and the
    receive rule (greedy.py:355-365: recipient r ANDs the set of every sender whose copy reached it) are applied here;
    the restatement then acts on the received sets with no message left to exchange."""
    nt = len(xy)
    seen = (np.asarray(empty_bits, dtype=np.int64) << np.arange(4)).sum(axis=-1)
    processed = np.asarray(memory['non_empty'], dtype=np.int64).copy()
    sends = (seen & processed) != 0
    processed[sends] &= ~seen[sends]
    delivered = np.ones((nt, nt), dtype=bool) if delivered is None else np.asarray(delivered, dtype=bool)
    received = processed.copy()
    for r in range(nt):
        for s in np.flatnonzero(sends & delivered[:, r]):
            received[r] &= processed[s]
    act, after = target_ref.team_step(xy, step_size, goal_bits, np.zeros_like(empty_bits, dtype=bool),
                                      dict(memory, non_empty=received), draws, noise_scale)
    after['sent'] = np.repeat(sends[:, None], nt, axis=1)
    return act, after


def camera_team_step(cam_xy, cam_phi, cam_theta, tgt_state, tracked, mem, draws, cfg, delivered=None):
    """``oracle.greedy_camera_ref.team_step`` with filtered messages.  A sent message is found by a delay draw no real
    draw reaches (the sender draws a delay for every message it sends); a dropped message is taken out by a pending
    delay of its sender towards the recipient, which leaves everything else of the step as it is; the senders' delays
    are those of the unfiltered step (the sender draws its delay whether or not the message arrives)."""
    nc = len(cam_xy)
    args = (cam_xy, cam_phi, cam_theta, tgt_state, tracked)
    sentinel = 1000   # > 2 * memory_period
    sent = camera_ref.team_step(*args, mem, dict(draws, delay=np.full((nc, nc), sentinel)), cfg)[1]['delay'] == sentinel
    act, after = camera_ref.team_step(*args, mem, draws, cfg)
    if delivered is not None:
        dropped = sent & ~np.asarray(delivered, dtype=bool)
        delay = np.where(dropped, 2.0, mem['delay'])   # the step first counts it down to 1: the message is not sent
        act, filtered = camera_ref.team_step(*args, dict(mem, delay=delay), draws, cfg)
        filtered['delay'] = after['delay']
        after = filtered
    after['sent'] = sent
    return act, after


# ---------------------------------------------------------------------------------------------------------------------
# fixtures shared with tests/test_agents.py (recorded reference agents)
# ---------------------------------------------------------------------------------------------------------------------
def _target_inputs(g, i):
    nt = int(g['cfg_counts'][1])
    goal_bits = np.zeros((nt, 4))
    for t in range(nt):
        if g['g_tgt_goal'][i][t] >= 0:
            goal_bits[t, g['g_tgt_goal'][i][t]] = g['g_tgt_goal_weight'][i][t]
    memory = {'goal': g['g_agent_goal_before'][i], 'non_empty': g['g_agent_non_empty_before'][i],
              'prev_xy': g['g_agent_prev_xy_before'][i], 'prev_noise': g['g_agent_prev_noise_before'][i]}
    draws = {'binomial': g['g_draw_binomial'][i], 'sample': g['g_draw_sample'][i], 'choice': g['g_draw_choice'][i]}
    return goal_bits, memory, draws


def _target_step(g, i, delivered=None):
    goal_bits, memory, draws = _target_inputs(g, i)
    step = float(g['cfg_target'][0])
    return target_team_step(g['g_tgt_xy'][i], step / g['g_tgt_capacity'][i], goal_bits,
                                       g['g_tgt_empty_bits'][i].astype(bool), memory, draws, float(g['noise_scale']),
                                       delivered=delivered)


def _camera_inputs(g, i):
    nt = int(g['cfg_counts'][1])
    loaded = (g['g_tgt_goal'][i] >= 0) & (g['g_tgt_goal_weight'][i] > 0)
    tgt_state = np.c_[g['g_tgt_xy'][i], np.full(nt, g['cfg_target'][1]), loaded.astype(float)]
    mem = {'memory': g['g_cam_mem_before'][i], 'time2forget': g['g_cam_time2forget_before'][i],
           'never_loaded': g['g_cam_never_loaded_before'][i], 'prev_action': g['g_cam_prev_action_before'][i],
           'delay': g['g_cam_delay_before'][i], 'neighbors': g['g_cam_neighbors_before'][i],
           'has_state': g['g_cam_has_state_message_before'][i]}
    draws = {'binomial': g['g_cam_draw_binomial'][i], 'sample': g['g_cam_draw_sample'][i], 'delay': g['g_cam_draw_delay'][i]}
    return tgt_state, mem, draws


def _camera_step(g, i, delivered=None):
    tgt_state, mem, draws = _camera_inputs(g, i)
    cam = g['cfg_camera']
    return camera_team_step(g['g_cam_xy'][i], g['g_cam_phi'][i], g['g_cam_theta'][i], tgt_state,
                                       g['g_mask_ct'][i].astype(bool), mem, draws, (cam[1], cam[2], cam[3], cam[4]),
                                       delivered=delivered)


def _pack_camera_memory(g, suffix):
    n, nc, nt = g['g_cam_mem' + suffix].shape[:3]
    return np.concatenate([
        g['g_cam_mem' + suffix].reshape(n, nc, 4 * nt), g['g_cam_time2forget' + suffix], g['g_cam_never_loaded' + suffix],
        g['g_cam_prev_action' + suffix], g['g_cam_delay' + suffix], g['g_cam_neighbors' + suffix][..., None],
        g['g_cam_has_state_message' + suffix][..., None]], axis=-1).astype(np.float64)


def _unpack(bits, n):
    """[B] int64 bit matrices (bit 8 s + r) -> [B, N, N] bool."""
    bits = np.asarray(bits).astype(np.uint64)
    shift = (8 * np.arange(n)[:, None] + np.arange(n)[None, :]).astype(np.uint64)
    return ((bits[:, None, None] >> shift) & np.uint64(1)).astype(bool)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: restatements
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', AGENT_NAMES + ['agents_Navigation'])
def test_restatements_with_every_message_delivered_reproduce_the_reference_agents(name):
    g = gu.load(name)
    nc, nt = int(g['cfg_counts'][0]), int(g['cfg_counts'][1])
    for i in range(int(g['count'])):
        act, after = _target_step(g, i, delivered=np.ones((nt, nt), dtype=bool))
        np.testing.assert_allclose(act, g['g_tgt_act'][i], rtol=0, atol=1e-12)
        np.testing.assert_array_equal(after['goal'], g['g_agent_goal_after'][i])
        np.testing.assert_array_equal(after['non_empty'], g['g_agent_non_empty_after'][i])
        np.testing.assert_allclose(after['prev_noise'], g['g_agent_prev_noise_after'][i], rtol=0, atol=1e-12)
        if nc == 0:
            continue
        act, after = _camera_step(g, i, delivered=np.ones((nc, nc), dtype=bool))
        np.testing.assert_allclose(act, g['g_cam_act'][i], rtol=0, atol=1e-9)
        np.testing.assert_array_equal(after['time2forget'], g['g_cam_time2forget_after'][i])
        np.testing.assert_array_equal(after['never_loaded'], g['g_cam_never_loaded_after'][i])
        np.testing.assert_array_equal(after['delay'], g['g_cam_delay_after'][i])
        np.testing.assert_array_equal(after['neighbors'], g['g_cam_neighbors_after'][i])
        np.testing.assert_allclose(after['memory'], g['g_cam_mem_after'][i], rtol=0, atol=1e-12)


def test_a_target_that_receives_nothing_keeps_its_own_set():
    xy = np.array([[0.0, 0.0], [100.0, 0.0], [0.0, 100.0]])
    empty = np.zeros((3, 4), dtype=bool)
    empty[0, 0] = True        # target 0 finds warehouse 0 empty: it broadcasts {1, 2, 3}
    empty[1, 1] = True        # target 1 finds warehouse 1 empty: it broadcasts {0, 2, 3}
    memory = {'goal': np.full(3, -1), 'non_empty': np.full(3, 15), 'prev_xy': xy.copy(), 'prev_noise': np.zeros((3, 2))}
    draws = {'binomial': np.zeros(3, dtype=bool), 'sample': np.zeros((3, 2)), 'choice': np.array([3, 3, 3])}
    args = (xy, np.full(3, 10.0), np.zeros((3, 4)), empty, memory, draws, 0.5)
    _, every = target_team_step(*args)
    assert every['non_empty'].tolist() == [12, 12, 12]
    assert every['sent'].tolist() == [[True] * 3, [True] * 3, [False] * 3]
    _, none = target_team_step(*args, delivered=np.zeros((3, 3), dtype=bool))
    assert none['non_empty'].tolist() == [14, 13, 15]
    only_own = np.eye(3, dtype=bool)
    _, own = target_team_step(*args, delivered=only_own)
    assert own['non_empty'].tolist() == [14, 13, 15]
    within = delivered_in_range(xy, 100.0)
    assert within.tolist() == [[True, True, True], [True, True, False], [True, False, True]]
    _, ranged = target_team_step(*args, delivered=within)
    assert ranged['non_empty'].tolist() == [12, 12, 14]


def test_a_dropped_camera_state_message_sets_the_delay_but_not_the_neighbour():
    nc, nt = 2, 1
    mem = {'memory': np.zeros((nc, nt, 4)), 'time2forget': np.zeros((nc, nt)), 'never_loaded': np.ones((nc, nt)),
           'prev_action': np.zeros((nc, 2)), 'delay': np.zeros((nc, nc)), 'neighbors': np.zeros(nc, dtype=np.int64),
           'has_state': np.ones(nc, dtype=np.int64)}
    draws = {'binomial': np.zeros(nc), 'sample': np.zeros((nc, 2)), 'delay': np.array([[0, 17], [9, 0]])}
    args = (np.array([[0.0, 0.0], [1000.0, 0.0]]), np.zeros(nc), np.full(nc, 90.0), np.array([[500.0, 500.0, 500.0, 0.0]]),
            np.zeros((nc, nt), dtype=bool), mem, draws, (15.0, 1500.0, 5.0, 2.5))
    _, every = camera_team_step(*args)
    assert every['neighbors'].tolist() == [2, 1] and every['sent'].tolist() == [[False, True], [True, False]]
    delivered = np.array([[False, False], [True, False]])   # camera 0's message to camera 1 is dropped
    _, after = camera_team_step(*args, delivered=delivered)
    assert after['neighbors'].tolist() == [2, 0]
    assert after['delay'].tolist() == [[0, 17], [9, 0]] and after['has_state'].tolist() == [0, 0]


# ---------------------------------------------------------------------------------------------------------------------
# CPU: single-environment mode on a recorded simulator
# ---------------------------------------------------------------------------------------------------------------------
class FilterRecordingSim:
    """Recorded observations of ``wrappers_4v8-9.npz`` (``ObservationsOnlySim``) plus the filter registration."""

    filters = []

    @classmethod
    def make(cls):
        from test_reference_wrappers import ObservationsOnlySim  # pylint: disable=import-outside-toplevel

        class Sim(ObservationsOnlySim):
            B = 1

            def set_message_filter(self, **kwargs):
                cls.filters.append(kwargs)

        return Sim


@pytest.fixture()
def single_env():
    import mate_b200.environment as b200  # pylint: disable=import-outside-toplevel

    g = np.load(os.path.join(GOLDEN, 'wrappers_4v8-9.npz'))
    sim = FilterRecordingSim.make()
    sim.fixture = (g, 'w_')
    FilterRecordingSim.filters.clear()
    env_class = type('MultiAgentTracking', (b200.MultiAgentTracking,), {'_sim_class': sim})
    env = env_class(config=str(g['config_name']))
    env.reset()
    return env, g


def _broadcast_all(env, Message, Team):
    for team, n in ((Team.CAMERA, env.num_cameras), (Team.TARGET, env.num_targets)):
        for s in range(n):
            env.send_messages(Message(sender=s, recipient=None, content={'s': s}, team=team))


def _received(base):
    cams, tgts = base.receive_messages()
    out = []
    for inbox, n in ((cams, base.num_cameras), (tgts, base.num_targets)):
        got = np.zeros((n, n), dtype=bool)
        for r, messages in enumerate(inbox):
            for m in messages:
                assert m.recipient == r
                got[m.sender, r] = True
        out.append(got)
    return out


def test_single_env_range_filter_on_the_recorded_positions(single_env):
    import mate_b200 as mate  # pylint: disable=import-outside-toplevel

    base, g = single_env
    limit = 1000.0
    env = mate.RestrictedCommunicationRange(base, range_limit=limit)
    assert FilterRecordingSim.filters[-1]['range_limit'] == (limit, limit)
    assert FilterRecordingSim.filters[-1]['keep_probability'] == (1.0, 1.0)
    _broadcast_all(env, mate.Message, mate.Team)
    cams, tgts = _received(base)
    want_cams = delivered_in_range(g['w_cam_xy'][0], limit)
    want_tgts = delivered_in_range(g['w_tgt_xy'][0], limit)
    assert not want_cams.all() and want_cams.any()        # the limit cuts some pairs and keeps others
    np.testing.assert_array_equal(cams, want_cams)
    np.testing.assert_array_equal(tgts, want_tgts)
    assert (base.camera_communication_edges == want_cams).all()
    # peer-to-peer messages go through the same rule
    env.send_messages([mate.Message(sender=0, recipient=r, content=None, team=mate.Team.CAMERA) for r in range(base.num_cameras)])
    cams, _ = _received(base)
    np.testing.assert_array_equal(cams[0], want_cams[0])


@pytest.mark.parametrize('rate', [0.0, 1.0])
def test_single_env_dropout_rates_zero_and_one(single_env, rate):
    import mate_b200 as mate  # pylint: disable=import-outside-toplevel

    base, _ = single_env
    env = mate.RandomMessageDropout(base, dropout_rate=rate)
    assert FilterRecordingSim.filters[-1]['keep_probability'] == (1.0 - rate, 1.0 - rate)
    _broadcast_all(env, mate.Message, mate.Team)
    cams, tgts = _received(base)
    assert cams.all() and tgts.all() if rate == 0.0 else not (cams.any() or tgts.any())
    assert int(base.target_communication_edges.sum()) == (base.num_targets ** 2 if rate == 0.0 else 0)


def test_single_env_stacked_dropouts_keep_the_product(single_env):
    import mate_b200 as mate  # pylint: disable=import-outside-toplevel

    base, _ = single_env
    env = mate.RestrictedCommunicationRange(mate.RandomMessageDropout(mate.RandomMessageDropout(base, 0.25), 0.5), range_limit=1500)
    assert FilterRecordingSim.filters[-1]['keep_probability'] == (0.375, 0.375)
    assert FilterRecordingSim.filters[-1]['range_limit'] == (1500.0, 1500.0)
    assert str(env).startswith('<RestrictedCommunicationRange<RandomMessageDropout<RandomMessageDropout')


@pytest.mark.parametrize('team', ['camera', 'target', 'both', 'none'])
def test_single_env_no_communication_per_team(single_env, team):
    import mate_b200 as mate  # pylint: disable=import-outside-toplevel

    base, _ = single_env
    env = mate.NoCommunication(base, team=team)
    camera_off, target_off = team in ('camera', 'both'), team in ('target', 'both')
    assert FilterRecordingSim.filters[-1]['keep_probability'] == (0.0 if camera_off else 1.0, 0.0 if target_off else 1.0)
    _broadcast_all(env, mate.Message, mate.Team)
    cams, tgts = _received(base)
    assert cams.all() != camera_off and not (camera_off and cams.any())
    assert tgts.all() != target_off and not (target_off and tgts.any())
    env.step((np.zeros((base.num_cameras, 2)), np.zeros((base.num_targets, 2))))
    assert int(base.camera_total_communication_edges.sum()) == (0 if camera_off else base.num_cameras ** 2)


def test_a_communication_wrapper_above_a_single_team_wrapper_fails(single_env):
    import mate_b200 as mate  # pylint: disable=import-outside-toplevel

    base, _ = single_env
    below = mate.MultiTarget(mate.RandomMessageDropout(base, 0.25), camera_agent=mate.GreedyCameraAgent(seed=0))
    assert isinstance(below.env, mate.RandomMessageDropout)
    for wrap in (lambda e: mate.RestrictedCommunicationRange(e, range_limit=10.0), lambda e: mate.RandomMessageDropout(e, 0.5),
                 lambda e: mate.NoCommunication(e, team='both')):
        for single_team in (mate.MultiTarget(base, camera_agent=mate.GreedyCameraAgent(seed=0)),
                            mate.MultiCamera(base, target_agent=mate.GreedyTargetAgent(seed=0))):
            with pytest.raises(AssertionError, match='before `MultiCamera` / `MultiTarget`'):
                wrap(single_team)


def test_invalid_wrapper_arguments():
    import mate_b200 as mate  # pylint: disable=import-outside-toplevel

    with pytest.raises(AssertionError):
        mate.RandomMessageDropout(None, 1.5)
    with pytest.raises(AssertionError):
        mate.RestrictedCommunicationRange(None, -1.0)
    with pytest.raises(AssertionError):
        mate.NoCommunication(None, team='cameras')


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _golden_sim(g):
    from mate_b200.sim import BatchedSim  # pylint: disable=import-outside-toplevel

    n = int(g['count'])
    sim = BatchedSim(gu.flat_config(g), n, device=0)
    sim.set_state(gu.stack_states([gu.state_arrays(g, 'g_', i) for i in range(n)]))
    return sim


def _edge_tensors(sim):
    delivered = tuple(torch.zeros(sim.B, dtype=torch.int64, device=sim.device) for _ in range(2))
    totals = tuple(torch.zeros((sim.B, n, n), dtype=torch.int32, device=sim.device) for n in (sim.nc, sim.nt))
    return delivered, totals


def _golden_target_call(g, sim, agent):
    memory = np.concatenate([g['g_agent_goal_before'][..., None], g['g_agent_non_empty_before'][..., None],
                             g['g_agent_prev_xy_before'], g['g_agent_prev_noise_before']], axis=-1).astype(np.float64)
    agent.memory.copy_(torch.from_numpy(memory))
    actions = agent.act(replay={'binomial': g['g_draw_binomial'], 'sample': g['g_draw_sample'], 'choice': g['g_draw_choice']})
    torch.cuda.synchronize()
    return actions.cpu().numpy(), agent.memory.cpu().numpy()


def _golden_camera_call(g, sim, agent):
    agent.memory.copy_(torch.from_numpy(_pack_camera_memory(g, '_before')))
    actions = agent.act(g['g_mask_ct'], replay={'binomial': g['g_cam_draw_binomial'], 'sample': g['g_cam_draw_sample'],
                                                'delay': g['g_cam_draw_delay']})
    torch.cuda.synchronize()
    return actions.cpu().numpy(), agent.memory.cpu().numpy()


def _near_ties(xy, limit):
    xy = np.asarray(xy, dtype=np.float64)
    d = np.sqrt(((xy[:, :, None, :] - xy[:, None, :, :]) ** 2).sum(-1))
    return np.abs(d - limit) <= NEAR_TIE * limit


@pytest.mark.gpu
@pytest.mark.parametrize('name', AGENT_NAMES)
@pytest.mark.parametrize('limits,keep', [((800.0, 100.0), 1.0), ((1500.0, 300.0), 1.0), ((1500.0, 300.0), 0.7)])
def test_kernels_against_the_restatements_with_filters(name, limits, keep):
    """Range (per team: cameras, targets) and dropout on recorded states with replayed agent draws: the kernels'
    delivered bits are the sent messages within range (all of them without dropout, a subset with it), and feeding
    them into the restatements reproduces the kernels' memory and actions."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    g = gu.load(name)
    n, nc, nt = int(g['count']), int(g['cfg_counts'][0]), int(g['cfg_counts'][1])
    sim = _golden_sim(g)
    delivered, totals = _edge_tensors(sim)
    sim.set_message_filter(range_limit=limits, keep_probability=(keep, keep), delivered=delivered, total_edges=totals)
    targets = mate_b200.GreedyTargetAgent(seed=1, noise_scale=float(g['noise_scale']))
    cameras = mate_b200.GreedyCameraAgent(seed=1)
    targets.bind(sim)
    cameras.bind(sim)
    cut = {0: 0, 1: 0}
    for team, call, step, xy_key, size in ((1, _golden_target_call, _target_step, 'g_tgt_xy', nt),
                                           (0, _golden_camera_call, _camera_step, 'g_cam_xy', nc)):
        actions, memory = call(g, sim, targets if team == 1 else cameras)
        bits = _unpack(delivered[team].cpu().numpy(), size)
        np.testing.assert_array_equal(totals[team].cpu().numpy(), bits.astype(np.int32))   # first call: no reset, totals were zero
        ties = _near_ties(g[xy_key], limits[team])
        for i in range(n):
            sent = step(g, i)[1]['sent']
            want = sent & delivered_in_range(g[xy_key][i], limits[team])
            cut[team] += int((sent & ~want).sum())
            got = bits[i]
            if keep == 1.0:
                np.testing.assert_array_equal(got[~ties[i]], want[~ties[i]], err_msg=f'team {team} sample {i}')
            else:
                assert not (got & ~(want | ties[i])).any(), f'team {team} sample {i}'
            act, after = step(g, i, delivered=got)
            np.testing.assert_allclose(actions[i], act, rtol=1e-6, atol=1e-5)
            if team == 1:
                np.testing.assert_array_equal(memory[i, :, 0], after['goal'])
                np.testing.assert_array_equal(memory[i, :, 1], after['non_empty'])
                np.testing.assert_allclose(memory[i, :, 4:6], after['prev_noise'], rtol=0, atol=1e-12)
            else:
                np.testing.assert_allclose(memory[i, :, :4 * nt], after['memory'].reshape(nc, 4 * nt), rtol=0, atol=1e-12)
                np.testing.assert_array_equal(memory[i, :, 4 * nt:5 * nt], after['time2forget'])
                np.testing.assert_array_equal(memory[i, :, 5 * nt:6 * nt], after['never_loaded'])
                np.testing.assert_array_equal(memory[i, :, 6 * nt + 2:6 * nt + 2 + nc], after['delay'])
                np.testing.assert_array_equal(memory[i, :, 6 * nt + 2 + nc], after['neighbors'])
    assert cut[0] > 0   # the camera limits cut sent messages
    sim.close()


@pytest.mark.gpu
@pytest.mark.parametrize('name', AGENT_NAMES)
def test_no_deliveries_match_the_restatements(name):
    """NoCommunication for both teams on recorded states: nothing is delivered, and the memories equal the restatements
    with no deliveries."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    g = gu.load(name)
    n, nc, nt = int(g['count']), int(g['cfg_counts'][0]), int(g['cfg_counts'][1])
    sim = _golden_sim(g)
    delivered, totals = _edge_tensors(sim)
    sim.set_message_filter(keep_probability=(0.0, 0.0), delivered=delivered, total_edges=totals)
    targets = mate_b200.GreedyTargetAgent(seed=1, noise_scale=float(g['noise_scale']))
    cameras = mate_b200.GreedyCameraAgent(seed=1)
    targets.bind(sim)
    cameras.bind(sim)
    t_act, t_mem = _golden_target_call(g, sim, targets)
    c_act, c_mem = _golden_camera_call(g, sim, cameras)
    assert int(delivered[0].abs().sum()) == 0 and int(delivered[1].abs().sum()) == 0
    assert int(totals[0].sum()) == 0 and int(totals[1].sum()) == 0
    for i in range(n):
        act, after = _target_step(g, i, delivered=np.zeros((nt, nt), dtype=bool))
        np.testing.assert_allclose(t_act[i], act, rtol=1e-6, atol=1e-5)
        np.testing.assert_array_equal(t_mem[i, :, 1], after['non_empty'])
        act, after = _camera_step(g, i, delivered=np.zeros((nc, nc), dtype=bool))
        np.testing.assert_allclose(c_act[i], act, rtol=1e-6, atol=1e-5)
        np.testing.assert_array_equal(c_mem[i, :, 6 * nt + 2 + nc], after['neighbors'])
        np.testing.assert_array_equal(c_mem[i, :, 6 * nt + 2:6 * nt + 2 + nc], after['delay'])
    sim.close()


def _single_team_run(wrap_comm, team, steps, num_envs=64, seed=3, agent_seed=5, config='MATE-4v8-9.yaml', **cfg):
    """Run MultiCamera (team 0 learns, greedy targets) or MultiTarget (team 1 learns, greedy cameras) with zero actions;
    per step: opponent actions, opponent memory, delivered bits and totals of the opponent team."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    def single_team(e):
        e = wrap_comm(e)
        if team == 0:
            return mate_b200.MultiCamera(e, target_agent=mate_b200.GreedyTargetAgent(seed=agent_seed))
        return mate_b200.MultiTarget(e, camera_agent=mate_b200.GreedyCameraAgent(seed=agent_seed))

    env = mate_b200.make('MultiAgentTracking-v0', config=config, num_envs=num_envs, wrappers=[single_team], **cfg)
    env.reset(seed=seed)
    base = env.unwrapped
    n = base.num_cameras if team == 0 else base.num_targets
    zeros = torch.zeros((num_envs, n, 2), device='cuda')
    out = []
    for _ in range(steps):
        env.step(zeros)
        out.append(_record(env, team))
    return env, out


def _record(env, team):
    base = env.unwrapped
    opponent = 1 - team
    return (env.opponent_agent.actions.cpu().numpy().copy(), env.opponent_agent.memory.cpu().numpy().copy(),
            base._delivered_bits[opponent].cpu().numpy().copy(),   # pylint: disable=protected-access
            base.total_communication_edges[opponent].cpu().numpy().copy())


@pytest.mark.gpu
@pytest.mark.parametrize('team', [0, 1])
def test_an_unrestricted_filter_changes_nothing(team):
    """No filter at all (the simulator's default) against registered wrappers that restrict nothing, 200 live steps:
    actions and memory bitwise equal; the edges are counted either way."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    def unregistered(e):
        e.unwrapped.sim.set_message_filter()
        return e

    def unrestricted(e):
        return mate_b200.NoCommunication(mate_b200.RandomMessageDropout(mate_b200.RestrictedCommunicationRange(e, np.inf), 0.0), 'none')

    env_a, plain = _single_team_run(unregistered, team, 200)
    env_b, wrapped = _single_team_run(unrestricted, team, 200)
    for (act_a, mem_a, bits_a, _), (act_b, mem_b, bits_b, tot_b) in zip(plain, wrapped):
        np.testing.assert_array_equal(act_a, act_b)
        np.testing.assert_array_equal(mem_a, mem_b)
        assert (bits_a == 0).all()
    assert sum(int((bits != 0).sum()) for _, _, bits, _ in wrapped) > 0
    env_a.close()
    env_b.close()


def _popcount(bits):
    bits = bits.view(-1, 1)
    return int(((bits >> torch.arange(64, device=bits.device)) & 1).sum())


@pytest.mark.gpu
@pytest.mark.parametrize('keep', [0.75, 0.1, 0.375])
def test_dropout_statistics(keep):
    """65 536 environments of MATE-4v8-9 over 50 steps (after 200 to settle): every call runs twice on the same memory and serial, without
    a filter (the sent messages) and with dropout; the delivered messages are a subset of the sent ones and their
    fraction lies within 5 sigma of the keep probability (0.375 = two stacked dropouts of 0.25 and 0.5)."""
    import mate_b200  # pylint: disable=import-outside-toplevel
    from mate_b200.config import flatten_config, read_config  # pylint: disable=import-outside-toplevel
    from mate_b200.sim import BatchedSim  # pylint: disable=import-outside-toplevel

    B = 65536
    sim = BatchedSim(flatten_config(read_config('MATE-4v8-9.yaml')), B, device=0)
    sim.reset(seed=4)
    sim.observe(aux=True)
    delivered, totals = _edge_tensors(sim)
    targets, cameras = mate_b200.GreedyTargetAgent(seed=2), mate_b200.GreedyCameraAgent(seed=3)
    targets.bind(sim)
    cameras.bind(sim)
    sent_n, kept_n = [0, 0], [0, 0]
    reset = True
    for _ in range(200):   # targets broadcast once they find empty warehouses: settle first
        tracked = (sim.cam_obs[..., 26:22 + 5 * 8:5] > 0.5).to(torch.uint8)
        tgt_act, cam_act = targets.act(reset_mask=reset).clone(), cameras.act(tracked, reset_mask=reset).clone()
        reset = None
        sim.step(cam_act, tgt_act, auto_reset=True, aux=True)
    for _ in range(50):
        tracked = (sim.cam_obs[..., 26:22 + 5 * 8:5] > 0.5).to(torch.uint8)
        acts = []
        for team, agent, call in ((1, targets, lambda a, r: a.act(reset_mask=r)), (0, cameras, lambda a, r: a.act(tracked, reset_mask=r))):
            memory, serial = agent._memory.clone(), agent._serial   # pylint: disable=protected-access
            sim.set_message_filter(delivered=delivered, total_edges=totals)
            call(agent, reset)
            sent = delivered[team].clone()
            agent._memory.copy_(memory)   # pylint: disable=protected-access
            agent._serial = serial        # pylint: disable=protected-access
            sim.set_message_filter(keep_probability=(keep, keep), delivered=delivered, total_edges=totals)
            acts.append(call(agent, reset).clone())
            kept = delivered[team]
            assert int((kept & ~sent).abs().sum()) == 0
            sent_n[team] += _popcount(sent)
            kept_n[team] += _popcount(kept)
        reset = None
        sim.step(acts[1], acts[0], auto_reset=True, aux=True)
    for team in range(2):
        n = sent_n[team]
        assert n > 1000, (team, n)
        sigma = np.sqrt(n * keep * (1 - keep))
        assert abs(kept_n[team] - n * keep) <= 5 * sigma, (team, kept_n[team], n * keep, sigma)
    sim.close()


@pytest.mark.gpu
def test_filtered_draws_do_not_depend_on_the_batch_split():
    """128 environments against 64 + 64 (env_index_base 64) under range + dropout: delivered bits, totals, actions and
    memory bitwise equal; the drops differ across steps and agree for the same seed."""
    import mate_b200  # pylint: disable=import-outside-toplevel
    from mate_b200.config import flatten_config, read_config  # pylint: disable=import-outside-toplevel
    from mate_b200.sim import BatchedSim  # pylint: disable=import-outside-toplevel

    cfg = flatten_config(read_config('MATE-4v8-9.yaml'))

    def run(num_envs, base, seed=9):
        sim = BatchedSim(cfg, num_envs, device=0, env_index_base=base)
        sim.reset(seed=seed)
        sim.observe(aux=True)
        delivered, totals = _edge_tensors(sim)
        sim.set_message_filter(range_limit=(1500.0, 300.0), keep_probability=(0.5, 0.5), delivered=delivered, total_edges=totals)
        targets, cameras = mate_b200.GreedyTargetAgent(seed=5), mate_b200.GreedyCameraAgent(seed=6)
        targets.bind(sim)
        cameras.bind(sim)
        out = []
        reset = True
        for _ in range(40):
            tracked = (sim.cam_obs[..., 26:22 + 5 * 8:5] > 0.5).to(torch.uint8)
            tgt_act = targets.act(reset_mask=reset).clone()
            cam_act = cameras.act(tracked, reset_mask=reset).clone()
            reset = None
            sim.step(cam_act, tgt_act, auto_reset=True, aux=True)
            out.append([x.cpu().numpy().copy() for x in (cam_act, tgt_act, cameras._memory, targets._memory,   # pylint: disable=protected-access
                                                          delivered[0], delivered[1], totals[0], totals[1])])
        sim.close()
        return out

    whole, lo, hi, again = run(128, 0), run(64, 0), run(64, 64), run(128, 0)
    axes = [0, 0, 1, 2, 0, 0, 0, 0]   # environment axis of each recorded array
    for w, l, h, a in zip(whole, lo, hi, again):
        for k, axis in enumerate(axes):
            np.testing.assert_array_equal(w[k], np.concatenate([l[k], h[k]], axis=axis))
            np.testing.assert_array_equal(w[k], a[k])
    camera_bits = np.stack([w[4] for w in whole])
    assert len({row.tobytes() for row in camera_bits}) > 10   # the delivered sets change from step to step


@pytest.mark.gpu
def test_no_communication_of_the_opponent_team():
    """NoCommunication(team='camera') under MultiTarget: no camera message arrives and the cameras never learn of their
    teammates; team='target' under MultiCamera: no target message arrives."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    env, out = _single_team_run(lambda e: mate_b200.NoCommunication(e, team='camera'), 1, 60)
    nc, nt = 4, 8
    for _, memory, bits, totals in out:
        assert (bits == 0).all() and (totals == 0).all()
        assert (memory[..., 6 * nt + 2 + nc] == 0).all()
    env.close()
    env, out = _single_team_run(lambda e: mate_b200.NoCommunication(e, team='target'), 0, 60)
    for _, _, bits, totals in out:
        assert (bits == 0).all() and (totals == 0).all()
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize('team', [0, 1])
def test_totals_are_the_sum_since_the_agents_reset(team):
    """Per-episode totals equal the sum of the per-step delivered sets since the environment's agents were last reset,
    with auto-resets during the run (max_episode_steps=100)."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    def wrap(e):
        return mate_b200.RandomMessageDropout(e, 0.25)

    def single_team(e):
        e = wrap(e)
        if team == 0:
            return mate_b200.MultiCamera(e, target_agent=mate_b200.GreedyTargetAgent(seed=1))
        return mate_b200.MultiTarget(e, camera_agent=mate_b200.GreedyCameraAgent(seed=1))

    B = 1024
    env = mate_b200.make('MultiAgentTracking-v0', config='MATE-4v8-9.yaml', num_envs=B, max_episode_steps=100, wrappers=[single_team])
    env.reset(seed=2)
    base = env.unwrapped
    opponent = 1 - team
    n = (base.num_cameras, base.num_targets)[opponent]
    zeros = torch.zeros((B, (base.num_cameras, base.num_targets)[team], 2), device='cuda')
    expected = torch.zeros((B, n, n), dtype=torch.int32, device='cuda')
    resets = 0
    for _ in range(300):
        mask = env._reset_mask   # pylint: disable=protected-access
        mask = torch.ones(B, dtype=torch.bool, device='cuda') if mask is True else mask.bool()
        resets += int(mask.sum())
        env.step(zeros)
        expected = torch.where(mask.view(B, 1, 1), torch.zeros_like(expected), expected) + base.communication_edges[opponent].int()
        assert torch.equal(base.total_communication_edges[opponent], expected)
    assert resets > 2 * B   # the run crosses auto-resets
    assert int(expected.sum()) > 0
    env.close()


@pytest.mark.gpu
def test_snapshots_replay_drops_and_edges():
    """save_state / load_state(resume=True) through MultiTarget over the wrappers replays 50 steps bit for bit (camera
    actions, delivered bits, totals); a branched load carries the totals of the source environments."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    B = 128

    def comm(e):
        return mate_b200.RestrictedCommunicationRange(mate_b200.RandomMessageDropout(e, 0.25), range_limit=1500)

    env, _ = _single_team_run(comm, 1, 20, num_envs=B)
    zeros = torch.zeros((B, 8, 2), device='cuda')
    snapshot = env.save_state()
    saved_totals = env.unwrapped.total_communication_edges[0].clone()
    first = []
    for _ in range(50):
        env.step(zeros)
        first.append(_record(env, 1))
    env.load_state(snapshot, resume=True)
    assert torch.equal(env.unwrapped.total_communication_edges[0], saved_totals)
    for k in range(50):
        env.step(zeros)
        for a, b in zip(first[k], _record(env, 1)):
            np.testing.assert_array_equal(a, b)
    assert sum(int(r[3].sum()) for r in first) > 0
    src = np.arange(B)[::-1].copy()
    src[:4] = -1
    before = env.unwrapped.total_communication_edges[0].clone()
    env.load_state(snapshot, src=src)
    after = env.unwrapped.total_communication_edges[0]
    assert torch.equal(after[:4], before[:4])
    assert torch.equal(after[4:], saved_totals[torch.from_numpy(src[4:]).cuda()])
    env.close()


@pytest.mark.gpu
def test_message_filter_argument_checks():
    from mate_b200.config import flatten_config, read_config  # pylint: disable=import-outside-toplevel
    from mate_b200.sim import BatchedSim  # pylint: disable=import-outside-toplevel

    sim = BatchedSim(flatten_config(read_config('MATE-4v8-9.yaml')), 16, device=0)
    for kwargs in ({'range_limit': (-1.0, np.inf)}, {'range_limit': (np.nan, 1.0)}, {'keep_probability': (1.0, 1.5)},
                   {'keep_probability': (-0.1, 1.0)}, {'keep_probability': (np.nan, 1.0)}):
        with pytest.raises(ValueError):
            sim.set_message_filter(**kwargs)
    with pytest.raises(ValueError):
        sim.set_message_filter(delivered=(torch.zeros(15, dtype=torch.int64, device='cuda'), None))
    sim.set_message_filter(range_limit=(0.0, np.inf), keep_probability=(0.0, 1.0))
    sim.close()
