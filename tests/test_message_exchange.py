"""The tensor message channel of a learning team in batched mode (``MultiAgentTracking.exchange_messages``, C ABI
``mate_b200_exchange_messages``, DESIGN.md section 7i).

The kernel is checked against a NumPy restatement built here: the routed messages (the ``recipients`` mask or a
broadcast), the range rule of ``delivered_in_range`` (tests/test_communication_wrappers.py) on the positions of the
current state, and the inbox, sum and mean built from the delivered mask with a Python loop over the senders."""

import ctypes
import os
import re

import numpy as np
import pytest

from test_communication_wrappers import NEAR_TIE, FilterRecordingSim, GOLDEN, delivered_in_range

torch = pytest.importorskip('torch')

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REDUCTIONS = ('none', 'sum', 'mean')


# ---------------------------------------------------------------------------------------------------------------------
# the restatement
# ---------------------------------------------------------------------------------------------------------------------
def restate(content, sent, xy, range_limit=np.inf):
    """content float32 [B, N, D], sent bool [B, N(s), N(r)], xy float64 [B, N, 2] -> delivered [B, N(s), N(r)], the
    'none' inbox [B, N(r), N(s), D], the sum and the mean [B, N(r), D]."""
    delivered = sent & np.stack([delivered_in_range(xy[e], range_limit) for e in range(len(xy))])
    recipient_major = delivered.transpose(0, 2, 1)
    inbox = np.where(recipient_major[..., None], content[:, None, :, :], np.float32(0.0)).astype(np.float32)
    total = np.zeros((content.shape[0], content.shape[1], content.shape[2]), dtype=np.float32)
    for s in range(content.shape[1]):
        total = np.where(delivered[:, s, :, None], total + content[:, s, None, :], total)
    count = delivered.sum(axis=1).astype(np.float32)[..., None]
    with np.errstate(invalid='ignore', divide='ignore'):
        mean = np.where(count > 0, total / np.maximum(count, np.float32(1.0)), np.float32(0.0)).astype(np.float32)
    return delivered, {'none': inbox, 'sum': total, 'mean': mean}


def _near_ties(xy, limit):
    d = np.sqrt(((xy[:, :, None, :] - xy[:, None, :, :]) ** 2).sum(-1))
    return np.abs(d - limit) <= NEAR_TIE * limit


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _positions(env, team):
    return env.unwrapped.get_state()[('cam_xy', 'tgt_xy')[team]]


def _content(B, n, dim, seed):
    gen = torch.Generator(device='cuda')
    gen.manual_seed(seed)
    return torch.randn((B, n, dim), generator=gen, device='cuda') * 100.0


def _mask(B, n, seed, p=0.6):
    gen = torch.Generator(device='cuda')
    gen.manual_seed(seed)
    return torch.rand((B, n, n), generator=gen, device='cuda') < p


def _random_actions(env, k):
    base = env.unwrapped
    gen = torch.Generator(device='cuda')
    gen.manual_seed(500 + k)
    B, nc, nt = base.num_envs, base.num_cameras, base.num_targets
    cam = (torch.rand((B, nc, 2), generator=gen, device='cuda') * 2 - 1) * torch.tensor(
        [base.camera_rotation_step, base.camera_zooming_step], device='cuda') if nc else None
    tgt = (torch.rand((B, nt, 2), generator=gen, device='cuda') * 2 - 1) * base.target_step_size
    return cam, tgt


def _make(config, num_envs, wrap=None, **kwargs):
    import mate_b200  # pylint: disable=import-outside-toplevel

    env = mate_b200.make('MultiAgentTracking-v0', config=config, num_envs=num_envs, **kwargs)
    return wrap(env) if wrap is not None else env


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_header_message_codes_match_the_binding():
    from mate_b200 import _abi  # pylint: disable=import-outside-toplevel

    text = open(os.path.join(ROOT, 'include', 'mate_b200.h'), encoding='UTF-8').read()
    codes = {name: int(value) for name, value in re.findall(r'#define (MATE_MESSAGES_[A-Z]+) (\d+)', text)}
    assert codes == {'MATE_MESSAGES_NONE': _abi.MATE_MESSAGES_NONE, 'MATE_MESSAGES_SUM': _abi.MATE_MESSAGES_SUM,
                     'MATE_MESSAGES_MEAN': _abi.MATE_MESSAGES_MEAN}
    assert ctypes.sizeof(_abi.MateMessageExchange) == 5 * 8 + 4 * 4


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f'{name} was called: the arguments must be checked before any library call')


def _stand_in_sim(nc=4, nt=8, B=8):
    from mate_b200.sim import BatchedSim  # pylint: disable=import-outside-toplevel

    sim = BatchedSim.__new__(BatchedSim)   # no device: every check below has to happen on the host
    sim.B, sim.nc, sim.nt, sim.device, sim.lib, sim.handle = B, nc, nt, torch.device('cpu'), _NoLibrary(), None
    return sim


def test_arguments_are_checked_before_any_library_call():
    B, n, D = 8, 8, 5
    sim = _stand_in_sim()
    content = torch.zeros((B, n, D))
    mask = torch.zeros((B, n, n), dtype=torch.bool)
    episode = torch.full((B,), -1, dtype=torch.int32)
    good = dict(team=1, content=content, recipients=mask, reduction='none', serial=0, episode=episode)
    bad = [
        dict(team=2), dict(team=-1), dict(reduction='max'), dict(reduction=None),
        dict(content=content.double()), dict(content=content.half()), dict(content=content[:4]),
        dict(content=torch.zeros((B, n - 1, D))), dict(content=torch.zeros((B, n, 0))), dict(content=torch.zeros((B, n * D))),
        dict(content=torch.zeros((B, D, n)).transpose(1, 2)), dict(content=content.numpy()),
        dict(recipients=mask.float()), dict(recipients=mask.long()), dict(recipients=mask[:, :4]),
        dict(recipients=mask.transpose(1, 2)), dict(recipients=torch.zeros((B, n, n, 1), dtype=torch.bool)),
        dict(episode=episode.long()), dict(episode=episode[:4]), dict(episode=None),
        dict(team=0, content=torch.zeros((B, 4, D)), recipients=torch.zeros((B, 4, n), dtype=torch.bool)),
    ]
    for change in bad:
        with pytest.raises(ValueError):
            sim.exchange_messages(**dict(good, **change))
    # teams of 0 and of more than 8 agents
    for nc, nt, team in ((0, 8, 0), (4, 9, 1)):
        sim = _stand_in_sim(nc=nc, nt=nt)
        n = (nc, nt)[team]
        with pytest.raises(ValueError):
            sim.exchange_messages(team, torch.zeros((B, n, D)), None, 'none', 0, episode)


def test_single_environment_mode_raises():
    import mate_b200.environment as b200  # pylint: disable=import-outside-toplevel

    g = np.load(os.path.join(GOLDEN, 'wrappers_4v8-9.npz'))
    sim = FilterRecordingSim.make()
    sim.fixture = (g, 'w_')
    env = type('MultiAgentTracking', (b200.MultiAgentTracking,), {'_sim_class': sim})(config=str(g['config_name']))
    env.reset()
    with pytest.raises(NotImplementedError, match='send_messages'):
        env.exchange_messages('target', torch.zeros((1, 8, 4)))


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _check_call(env, team, content, mask, reduction, range_limit):
    """One exchange against the restatement: inbox, delivered, the delivered bits bitwise (near ties excluded)."""
    base = env.unwrapped
    xy = _positions(env, team)
    inbox, delivered = env.exchange_messages(team, content, mask, reduction=reduction)
    sent = np.ones(delivered.shape, dtype=bool) if mask is None else mask.cpu().numpy().astype(bool)
    want_delivered, want = restate(content.cpu().numpy(), sent, xy, range_limit)
    ties = _near_ties(xy, range_limit) if np.isfinite(range_limit) else np.zeros(sent.shape, dtype=bool)
    ok_pair = ~ties.transpose(0, 2, 1)                  # recipient-major
    ok_row = ok_pair.all(axis=2)                         # recipients without a near tie
    got_delivered = delivered.cpu().numpy()
    np.testing.assert_array_equal(got_delivered[ok_pair], want_delivered.transpose(0, 2, 1)[ok_pair])
    edges = base.communication_edges[team].cpu().numpy()
    np.testing.assert_array_equal(edges, got_delivered.transpose(0, 2, 1))
    got = inbox.cpu().numpy()
    if reduction == 'none':
        np.testing.assert_array_equal(got.view(np.int32)[ok_pair], want['none'].view(np.int32)[ok_pair])
    else:
        np.testing.assert_array_equal(got.view(np.int32)[ok_row], want[reduction].view(np.int32)[ok_row])
    return want_delivered


@pytest.mark.gpu
@pytest.mark.parametrize('config', ['MATE-4v8-9.yaml', 'MATE-4v2-0.yaml', 'MATE-8v8-9.yaml'])
def test_exact_against_the_restatement(config):
    """Both teams, random masks and broadcast, every reduction, D in {1, 5, 32}, a range limit that cuts pairs, keep = 1;
    the totals equal the sum of the delivered sets of the episode's exchanges."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    limit = 1000.0
    B = 512
    env = _make(config, B, wrap=lambda e: mate_b200.RestrictedCommunicationRange(e, limit))
    base = env.unwrapped
    env.reset(seed=11)
    for k in range(3):
        env.step(_random_actions(env, k))
    totals = [np.zeros((B, n, n), dtype=np.int32) for n in (base.num_cameras, base.num_targets)]
    cut, kept, call = 0, 0, 0
    for team, n in ((0, base.num_cameras), (1, base.num_targets)):
        for dim in (1, 5, 32):
            for reduction in REDUCTIONS:
                for broadcast in (False, True):
                    call += 1
                    content = _content(B, n, dim, call)
                    mask = None if broadcast else _mask(B, n, 100 + call)
                    delivered = _check_call(env, team, content, mask, reduction, limit)
                    sent = np.ones_like(delivered) if mask is None else mask.cpu().numpy()
                    cut += int((sent & ~delivered).sum())
                    kept += int(delivered.sum())
                    totals[team] += delivered
                    np.testing.assert_array_equal(base.total_communication_edges[team].cpu().numpy(), totals[team])
    assert cut > 0 and kept > 0
    env.close()


@pytest.mark.gpu
def test_nothing_delivered_and_undelivered_messages_are_not_read():
    """keep = 0 and NoCommunication on the team: nothing arrives, the inboxes are zeros even for NaN content and the
    totals do not change.  Without a filter, delivered is the send mask, and the NaN messages of senders that do not send
    to r never reach r's inbox or reduction."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    B, team, n, dim = 256, 1, 8, 8
    env = _make('MATE-4v8-9.yaml', B)
    env.reset(seed=3)
    mask = _mask(B, n, 7, p=0.5)
    content = _content(B, n, dim, 1)
    content[:, 0] = float('nan')   # sender 0's messages are NaN
    for reduction in REDUCTIONS:
        inbox, delivered = env.exchange_messages(team, content, mask, reduction)
        assert torch.equal(delivered, mask.transpose(1, 2))
        reached = mask[:, 0, :]   # [B, r]: sender 0 sends to r
        if reduction == 'none':
            assert not torch.isnan(inbox[:, :, 1:]).any()
            assert torch.isnan(inbox[:, :, 0]).any(dim=-1).eq(reached).all()
            assert (inbox[:, :, 0][~reached] == 0).all()
        else:
            assert torch.isnan(inbox).any(dim=-1).eq(reached).all()
    env.close()
    content = torch.full((B, n, dim), float('nan'), device='cuda')
    for wrap in (lambda e: mate_b200.RandomMessageDropout(e, 1.0), lambda e: mate_b200.NoCommunication(e, team='target')):
        env = _make('MATE-4v8-9.yaml', B)
        env.reset(seed=3)
        base = env.unwrapped
        env.exchange_messages(team, _content(B, n, dim, 2), mask)   # totals of the episode so far
        totals = base.total_communication_edges[team].clone()
        assert int(totals.sum()) > 0
        wrapped = wrap(env)
        for reduction in REDUCTIONS:
            for recipients in (None, mask):
                inbox, delivered = wrapped.exchange_messages('target', content, recipients, reduction)
                assert not delivered.any()
                assert (inbox.view(torch.int32) == 0).all()
                assert torch.equal(base.total_communication_edges[team], totals)
                assert not base.communication_edges[team].any()
        env.close()


@pytest.mark.gpu
@pytest.mark.parametrize('keep', [0.75, 0.1, 0.375])
def test_dropout_statistics(keep):
    """65 536 environments: delivered is a subset of sent, and the kept fraction lies within 5 sigma of the keep
    probability (0.375 = two stacked dropouts of 0.5 and 0.25)."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    def wrap(e):
        if keep == 0.375:
            return mate_b200.RandomMessageDropout(mate_b200.RandomMessageDropout(e, 0.5), 0.25)
        return mate_b200.RandomMessageDropout(e, 1.0 - keep)

    B = 65536
    env = _make('MATE-4v8-9.yaml', B, wrap=wrap)
    env.reset(seed=5)
    sent_n, kept_n = 0, 0
    for call in range(4):
        for team, n in ((0, 4), (1, 8)):
            mask = _mask(B, n, call * 2 + team) if call % 2 else None
            _, delivered = env.exchange_messages(team, _content(B, n, 1, call), mask)
            sent = torch.ones_like(delivered) if mask is None else mask.transpose(1, 2)
            assert not (delivered & ~sent).any()
            sent_n += int(sent.sum())
            kept_n += int(delivered.sum())
    sigma = np.sqrt(sent_n * keep * (1 - keep))
    assert abs(kept_n - sent_n * keep) <= 5 * sigma, (kept_n, sent_n * keep, sigma)
    env.close()


@pytest.mark.gpu
def test_draws_do_not_depend_on_the_batch_split():
    """128 environments against 64 + 64 (env_index_base 64) under range + dropout: bitwise equal inboxes, delivered
    masks and totals; the drops change from call to call."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    def run(num_envs, env_index_base, contents):
        env = _make('MATE-4v8-9.yaml', num_envs, env_index_base=env_index_base,
                    wrap=lambda e: mate_b200.RestrictedCommunicationRange(mate_b200.RandomMessageDropout(e, 0.5), 1200.0))
        env.reset(seed=9)
        lo = env_index_base
        out = []
        for k, (team, content) in enumerate(contents):
            if k % 3 == 2:
                env.step(tuple(None if a is None else a[lo:lo + num_envs] for a in _random_actions_for(128, k)))
            inbox, delivered = env.exchange_messages(team, content[lo:lo + num_envs].contiguous(), None, 'none')
            out.append([inbox.cpu().numpy(), delivered.cpu().numpy(), env.unwrapped.total_communication_edges[team].cpu().numpy()])
        env.close()
        return out

    contents = [(k % 2, _content(128, (4, 8)[k % 2], 4, k)) for k in range(12)]
    whole, low, high = run(128, 0, contents), run(64, 0, contents), run(64, 64, contents)
    for w, lo, hi in zip(whole, low, high):
        for a, b, c in zip(w, lo, hi):
            np.testing.assert_array_equal(a.view(np.uint8), np.concatenate([b, c]).view(np.uint8))
    target_sets = {w[1].tobytes() for (team, _), w in zip(contents, whole) if team == 1}
    assert len(target_sets) == 6   # every call draws anew


def _random_actions_for(B, k):
    gen = torch.Generator(device='cuda')
    gen.manual_seed(900 + k)
    cam = (torch.rand((B, 4, 2), generator=gen, device='cuda') * 2 - 1) * torch.tensor([10.0, 5.0], device='cuda')
    tgt = (torch.rand((B, 8, 2), generator=gen, device='cuda') * 2 - 1) * 20.0
    return cam, tgt


@pytest.mark.gpu
def test_totals_across_auto_resets():
    """max_episode_steps=100, none, one or two calls between steps: the totals are the sum of the delivered sets since
    each environment's current episode began."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    B, team, n = 1024, 1, 8
    env = _make('MATE-4v8-9.yaml', B, max_episode_steps=100,
                wrap=lambda e: mate_b200.RestrictedCommunicationRange(mate_b200.RandomMessageDropout(e, 0.25), 800.0))
    env.reset(seed=2)
    base = env.unwrapped
    expected = torch.zeros((B, n, n), dtype=torch.int32, device='cuda')
    fresh = torch.ones(B, dtype=torch.bool, device='cuda')   # no exchange yet in the environment's current episode
    resets = 0
    rng = np.random.RandomState(4)
    for k in range(260):
        for _ in range(int(rng.choice([0, 1, 1, 2]))):
            _, delivered = env.exchange_messages(team, _content(B, n, 2, k), _mask(B, n, k))
            expected = torch.where(fresh.view(B, 1, 1), torch.zeros_like(expected), expected) + delivered.transpose(1, 2).int()
            fresh.zero_()
            assert torch.equal(base.total_communication_edges[team], expected), k
        _, _, done, _ = env.step(_random_actions(env, k))
        fresh |= done
        resets += int(done.sum())
    assert resets > B and int(expected.sum()) > 0
    env.close()


def _exchanges(env, team, k, n, B):
    inbox, delivered = env.exchange_messages(team, _content(B, n, 4, k), _mask(B, n, k), 'sum' if k % 2 else 'none')
    return inbox.clone(), delivered.clone()


@pytest.mark.gpu
def test_snapshots_replay_the_exchanges():
    """save_state + load_state(resume=True) replays 50 steps of exchanges bit for bit (inbox, delivered, totals); a branched
    load carries the totals of the source environments and keeps the others'."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    B, team, n = 128, 1, 8
    env = _make('MATE-4v8-9.yaml', B, max_episode_steps=30,
                wrap=lambda e: mate_b200.RestrictedCommunicationRange(mate_b200.RandomMessageDropout(e, 0.25), 1500.0))
    env.reset(seed=8)
    base = env.unwrapped

    def run(first, last):
        out = []
        for k in range(first, last):
            inbox, delivered = _exchanges(env, team, k, n, B)
            env.step(_random_actions(env, k))
            out.append((inbox, delivered, base.total_communication_edges[team].clone()))
        return out

    run(0, 20)
    snapshot = env.save_state()
    saved_totals = base.total_communication_edges[team].clone()
    original = run(20, 70)
    env.load_state(snapshot, resume=True)
    assert torch.equal(base.total_communication_edges[team], saved_totals)
    for k, (want, got) in enumerate(zip(original, run(20, 70))):
        for a, b in zip(want, got):
            assert torch.equal(_bits(a), _bits(b)), k
    src = np.arange(B)[::-1].copy()
    src[:5] = -1
    before = base.total_communication_edges[team].clone()
    env.load_state(snapshot, src=src)
    after = base.total_communication_edges[team]
    assert torch.equal(after[:5], before[:5])
    assert torch.equal(after[5:], saved_totals[torch.from_numpy(src[5:]).cuda()])
    env.close()


@pytest.mark.gpu
def test_learning_targets_exchange_while_greedy_cameras_talk():
    """MultiTarget over RestrictedCommunicationRange(RandomMessageDropout(...)): the learning targets exchange tensors and
    the greedy cameras talk in their kernel; a resume replays both teams' traffic bit for bit."""
    import mate_b200  # pylint: disable=import-outside-toplevel

    B, n = 256, 8

    def single_team(e):
        e = mate_b200.RestrictedCommunicationRange(mate_b200.RandomMessageDropout(e, 0.25), range_limit=1500)
        return mate_b200.MultiTarget(e, camera_agent=mate_b200.GreedyCameraAgent(seed=5))

    env = mate_b200.make('MultiAgentTracking-v0', config='MATE-4v8-9.yaml', num_envs=B, max_episode_steps=40, wrappers=[single_team])
    env.reset(seed=3)
    base = env.unwrapped

    def run(first, last):
        out = []
        for k in range(first, last):
            inbox, delivered = _exchanges(env, 'target', k, n, B)
            env.step(_random_actions(env, k)[1])
            out.append((inbox, delivered, env.opponent_agent.actions.clone(), base._delivered_bits[0].clone(),   # pylint: disable=protected-access
                        base.total_communication_edges[0].clone(), base.total_communication_edges[1].clone()))
        return out

    run(0, 15)
    snapshot = env.save_state()
    original = run(15, 65)
    env.load_state(snapshot, resume=True)
    for k, (want, got) in enumerate(zip(original, run(15, 65))):
        for a, b in zip(want, got):
            assert torch.equal(_bits(a), _bits(b)), k
    assert sum(int(r[4].sum()) for r in original) > 0 and sum(int(r[5].sum()) for r in original) > 0
    env.close()


@pytest.mark.gpu
def test_the_channel_changes_nothing_else():
    """200 steps of MATE-4v8-9 with and without exchange calls: bitwise the same observations, rewards, done flags and
    state."""
    B = 512
    envs = [_make('MATE-4v8-9.yaml', B), _make('MATE-4v8-9.yaml', B)]
    for env in envs:
        env.reset(seed=21)
    for k in range(200):
        action = _random_actions(envs[0], k)
        team = k % 2
        n = (4, 8)[team]
        envs[1].exchange_messages(team, _content(B, n, 3, k), _mask(B, n, k) if k % 4 else None, REDUCTIONS[k % 3])
        outs = [env.step(action) for env in envs]
        (obs_a, rew_a, done_a, _), (obs_b, rew_b, done_b, _) = outs
        for a, b in zip(obs_a + rew_a, obs_b + rew_b):
            assert torch.equal(_bits(a), _bits(b)), k
        assert torch.equal(done_a, done_b), k
    state_a, state_b = (env.get_state() for env in envs)
    for name, value in state_a.items():
        np.testing.assert_array_equal(value, state_b[name], err_msg=name)
    for env in envs:
        env.close()


@pytest.mark.gpu
def test_abi_refusals_leave_the_handle_unchanged():
    from mate_b200 import _abi  # pylint: disable=import-outside-toplevel
    from mate_b200.config import flatten_config, read_config  # pylint: disable=import-outside-toplevel
    from mate_b200.sim import BatchedSim  # pylint: disable=import-outside-toplevel

    B, n, dim = 64, 8, 4
    sim = BatchedSim(flatten_config(read_config('MATE-4v8-9.yaml')), B, device=0)
    sim.reset(seed=1)
    lib = sim.lib
    content = _content(B, n, dim, 1)
    inbox = torch.full((B * n * n * dim + 4,), 7.0, device='cuda')
    delivered = torch.full((B * n * n + 4,), 3, dtype=torch.uint8, device='cuda')
    episode = torch.full((B,), 5, dtype=torch.int32, device='cuda')

    def call(**change):
        fields = dict(content=content.data_ptr(), recipients=None, inbox=inbox.data_ptr(), delivered=delivered.data_ptr(),
                      episode=episode.data_ptr(), team=1, dim=dim, reduction=_abi.MATE_MESSAGES_NONE, reserved=0)
        fields.update(change)
        x = _abi.MateMessageExchange(**fields)
        return lib.mate_b200_exchange_messages(sim.handle, ctypes.byref(x), 0, None)

    payload = sim.save_state().payload.clone()
    launches = sim.launch_count
    refusals = [dict(team=2), dict(team=-1), dict(dim=0), dict(dim=-3), dict(dim=1 << 30), dict(reduction=3), dict(reduction=-1),
                dict(content=None), dict(inbox=None), dict(episode=None), dict(content=content.data_ptr() + 2),
                dict(inbox=inbox.data_ptr() + 1), dict(episode=episode.data_ptr() + 2)]
    for change in refusals:
        assert call(**change) == -1, change   # MATE_EINVAL
        assert lib.mate_b200_last_error()
    assert lib.mate_b200_exchange_messages(None, None, 0, None) == -1
    torch.cuda.synchronize()
    assert sim.launch_count == launches
    assert (inbox == 7.0).all() and (delivered == 3).all() and (episode == 5).all()
    assert torch.equal(sim.save_state().payload, payload)
    sim.close()
    nav = BatchedSim(flatten_config(read_config('MATE-Navigation.yaml')), B, device=0)   # no cameras
    x = _abi.MateMessageExchange(content=content.data_ptr(), inbox=inbox.data_ptr(), episode=episode.data_ptr(), team=0, dim=dim)
    assert nav.lib.mate_b200_exchange_messages(nav.handle, ctypes.byref(x), 0, None) == -1
    nav.close()
