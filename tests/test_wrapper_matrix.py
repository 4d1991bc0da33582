"""The observation wrappers at every compiled shape, on every path that applies them, against a float64 restatement.

A wrapper registers op codes with the simulator; the rows are then transformed in one of three places, each with code
that changes with the (cameras, targets, obstacles) shape:
- the packer of the step kernel, for stacks ``(Enhanced | Shared)* Relative? Rescaled?`` whose rescale tables are
  uniform per entity kind (the folded fast path, ``pack_rows`` in ``mate_step.cuh``);
- the generic wrapper code on the staged rows (``apply_obs_ops``), for tables that are not uniform, or forced with
  ``MATE_B200_FOLD=0`` when the ops are set;
- a separate pass over the rows (``mate_b200_transform_observations``).
The independent side is ``oracle/obs_wrappers_ref.py``, a float64 NumPy restatement of the reference's wrappers that is
pinned to the reference's own output here (``tests/golden/wrappers_*.npz``).  On the GPU its input is the raw rows and
the state of a twin simulator without wrappers, driven identically; those raw rows are pinned to the float64 C oracle at
every shape by ``test_cuda_parity``.

Exactness: a copied entry, a flag, a zero and a relative coordinate are one fp64 value rounded once to float32 on both
sides, so they are compared bit for bit.  RescaledObservation is one float32 FMA with float32 (scale, shift) in the
library; its entries are compared with the float64 normalize_observation within what those roundings allow."""

import ctypes

import numpy as np
import pytest

import golden_util as gu
from oracle import obs_wrappers_ref as ref
from oracle.obs_wrappers_ref import ENHANCED_CAMERA as EN_C, ENHANCED_TARGET as EN_T, RELATIVE as REL, RESCALED as RESC
from oracle.obs_wrappers_ref import SHARED_CAMERA as SH_C, SHARED_TARGET as SH_T
from test_shape_matrix import SHAPES, _flat, _ids, preset_of

MASKS = (EN_C, EN_T, SH_C, SH_T)
PREFIXES = [()] + [(a,) for a in MASKS] + [(a, b) for a in MASKS for b in MASKS]   # mask prefixes of length 0 - 2
TAILS = [(), (REL,), (RESC,), (REL, RESC)]
FULL_MASKS = (SH_C, SH_T, SH_C, EN_C, SH_T, SH_C, SH_T, EN_T)    # 8 codes: fills the packed mask_ops word; the last one counts
SIX_MASKS_TAIL = (SH_T, EN_C, SH_C, SH_T, SH_C, SH_T, REL, RESC)
STACKS = [p + t for p in PREFIXES for t in TAILS] + [FULL_MASKS, SIX_MASKS_TAIL]
FORBIDDEN = [(REL, SH_C), (RESC, EN_T), (REL, RESC, SH_T), (REL, REL), (RESC, RESC), (RESC, REL), (SH_C, RESC, REL),
             (EN_C, REL, REL, RESC)]
NAMES = {EN_C: 'EN_C', EN_T: 'EN_T', SH_C: 'SH_C', SH_T: 'SH_T', REL: 'REL', RESC: 'RESC'}
GOLDEN = {   # the stacks of tests/test_wrappers.py (oracle/gen_wrapper_golden.py) as codes, camera codes kept
    'enhanced_both': (EN_C, EN_T), 'enhanced_camera': (EN_C,), 'enhanced_target': (EN_T,), 'shared_both': (SH_C, SH_T),
    'shared_camera': (SH_C,), 'shared_target': (SH_T,), 'relative': (REL,), 'rescaled': (RESC,),
    'shared_relative_rescaled': (SH_C, SH_T, REL, RESC), 'enhanced_relative_rescaled': (EN_C, EN_T, REL, RESC),
    'enhcam_sharedtgt_relative': (EN_C, SH_T, REL)}
LIMIT, SEED, ORACLE_ENVS, STEPS = 5, 23, 203, 3


def _name(ops):
    return ' '.join(NAMES[op] for op in ops) or '-'


# ------------------------------------------------------------------------------------------- the restatement pin (CPU)
def test_the_stack_enumeration():
    """21 mask prefixes x 4 tails, the 8-code mask stack and the 6 + 2 stack; every golden stack is among them."""
    from mate_b200 import _abi

    assert _abi.MAX_OBS_OPS == len(FULL_MASKS)
    assert len(PREFIXES) == 21 and len(STACKS) == 86 and len(set(STACKS)) == 86
    assert len(FULL_MASKS) == len(SIX_MASKS_TAIL) == 8 and set(FULL_MASKS) == set(MASKS)
    assert set(GOLDEN.values()) <= set(STACKS)


@pytest.mark.parametrize('name', sorted(GOLDEN))
def test_restatement_reproduces_the_reference(name):
    """CPU: the float64 restatement reproduces the reference's wrappers for every golden stack on every golden fixture,
    from the raw rows and the state the fixture holds."""
    from mate_b200 import _abi

    assert (ref.ENHANCED_CAMERA, ref.ENHANCED_TARGET, ref.SHARED_CAMERA, ref.SHARED_TARGET, ref.RELATIVE, ref.RESCALED) == \
        (_abi.OBS_ENHANCED_CAMERA, _abi.OBS_ENHANCED_TARGET, _abi.OBS_SHARED_CAMERA, _abi.OBS_SHARED_TARGET, _abi.OBS_RELATIVE,
         _abi.OBS_RESCALED)
    from test_wrappers import NAMES as fixtures

    assert len(fixtures) == 4
    for fixture in fixtures:
        g = gu.load(fixture)
        shape = tuple(int(x) for x in g['cfg_counts'])
        state = {'tgt_xy': g['w_tgt_xy'], 'cam_xy': g['w_cam_xy'], 'obs_xyr': g['w_obs_xyr'], 'remaining': g['w_remaining']}
        cam, tgt = ref.apply_ops(GOLDEN[name], g['w_cam_obs'], g['w_tgt_obs'], state, shape)
        assert cam.dtype == tgt.dtype == np.float64
        if shape[0]:
            assert np.abs(cam - g[f'w_{name}_cam_obs']).max() <= 1e-12, (fixture, name)
        assert np.abs(tgt - g[f'w_{name}_tgt_obs']).max() <= 1e-12, (fixture, name)


# ------------------------------------------------------------------------------------------------ fast-path guard (CPU)
def uniform_tables(shape):
    """The uniformity check of mate_b200_set_observation_ops over rescale_tables: the preserved columns are the same in
    both teams' rows, and every entry of a kind has one (scale, shift) in both teams' rows.  Only then does a stack with
    RescaledObservation run on the folded fast path."""
    from mate_b200.sim import rescale_tables

    nc, nt, no = shape
    cam_t, tgt_t = rescale_tables(nc, nt, no)
    ok = not nc or np.array_equal(cam_t[:ref.P], tgt_t[:ref.P])
    entry = {}
    for team, table in (('target', tgt_t), ('camera', cam_t)):
        if team == 'camera' and not nc:
            continue
        for kind, w, n, first in ref.blocks(team, shape):
            for e in range(n):
                cols = table[first + (w + 1) * e:first + (w + 1) * (e + 1)]
                entry.setdefault(kind, cols)
                ok = ok and np.array_equal(cols, entry[kind])
    return ok


@pytest.mark.parametrize('shape', SHAPES, ids=_ids(SHAPES))
def test_rescale_tables_keep_every_shape_on_the_fast_path(shape):
    """CPU: a table change that silently demoted a shape to the generic path would fail here."""
    assert uniform_tables(shape)


def test_the_fast_path_guard_sees_a_non_uniform_table(monkeypatch):
    """The guard is not vacuous: one entry column that differs between two targets breaks it."""
    from mate_b200 import sim as simmod

    real = simmod.rescale_tables

    def skewed(nc, nt, no):
        cam_t, tgt_t = real(nc, nt, no)
        return cam_t, _skew(tgt_t, (nc, nt, no))

    monkeypatch.setattr(simmod, 'rescale_tables', skewed)
    assert not uniform_tables((4, 8, 9))


def _skew(tgt_t, shape):
    """A copy of the target table whose x column differs between the entries of target 0 and target 1."""
    (_, w, _, first), = [b for b in ref.blocks('target', shape) if b[0] == 'tgt']
    out = tgt_t.copy()
    out[first + (w + 1), 0] *= 1.5
    out[first + (w + 1), 1] += 0.25
    return out


# ---------------------------------------------------------------------------------------------------- order rules (CPU)
class _FakeSim:
    def __init__(self):
        self._obs_ops = []

    def set_observation_wrappers(self, ops):
        from mate_b200.sim import check_observation_ops

        self._obs_ops = check_observation_ops(ops)


class _FakeEnv:   # what the observation wrappers' constructors read of the environment
    def __init__(self, shape):
        from mate_b200 import constants

        self.num_cameras, self.num_targets, self.num_obstacles = shape
        self.camera_observation_space = constants.camera_observation_space_of(*shape)
        self.target_observation_space = constants.target_observation_space_of(*shape)
        self.sim = _FakeSim()
        self.unwrapped = self


def _wrap(ops, shape=(4, 8, 9)):
    import mate_b200

    env = base = _FakeEnv(shape)
    for op in ops:
        if op in MASKS:
            cls = mate_b200.EnhancedObservation if op in (EN_C, EN_T) else mate_b200.SharedFieldOfView
            env = cls(env, team='camera' if op in (EN_C, SH_C) else 'target')
        else:
            env = (mate_b200.RelativeCoordinates if op == REL else mate_b200.RescaledObservation)(env)
    return base


@pytest.mark.parametrize('stack', STACKS, ids=[_name(s) for s in STACKS])
def test_every_enumerated_stack_is_accepted(stack):
    """CPU: the wrapper classes build every enumerated stack and register exactly its codes; so does the simulator's check."""
    from mate_b200.sim import check_observation_ops

    assert _wrap(stack).sim._obs_ops == list(stack)   # pylint: disable=protected-access
    assert check_observation_ops(stack) == list(stack)


@pytest.mark.parametrize('stack', FORBIDDEN, ids=[_name(s) for s in FORBIDDEN])
def test_forbidden_orders_are_refused(stack):
    """CPU: the orders the reference's assertions forbid -- a mask wrapper after RelativeCoordinates or RescaledObservation,
    either of those twice, RelativeCoordinates after RescaledObservation -- are refused by the wrapper classes
    (AssertionError, as in the reference) and by BatchedSim.set_observation_wrappers (ValueError) before any library call,
    which leaves the registered codes as they were."""
    from mate_b200.sim import BatchedSim, check_observation_ops

    with pytest.raises(AssertionError):
        _wrap(stack)
    with pytest.raises(ValueError):
        check_observation_ops(stack)
    sim = BatchedSim.__new__(BatchedSim)   # no library and no device: a library call would raise AttributeError
    sim._obs_ops = [SH_C, REL]             # pylint: disable=protected-access
    with pytest.raises(ValueError):
        sim.set_observation_wrappers(stack)
    assert sim._obs_ops == [SH_C, REL]     # pylint: disable=protected-access


def test_the_simulator_check_refuses_unknown_codes_and_long_stacks():
    from mate_b200.sim import check_observation_ops

    for bad in ([0], [7], [SH_C, -1], [SH_C] * 9):
        with pytest.raises(ValueError):
            check_observation_ops(bad)
    assert check_observation_ops([]) == [] and check_observation_ops(np.array([SH_T, REL])) == [SH_T, REL]


# --------------------------------------------------------------------------------------------------------- the edge batch
BLIND_ENV, CLUSTER_ENV, CORNER_ENVS = 0, 1, (2, 3)
EDGE_ENVS = 4
TRUE_EMPTY = (0b0101, 0b0010, 0b0000, 0b1111)   # per edge environment: the warehouses with no cargo left


def edge_states(cfg, seed=11):
    """A constructed batch of EDGE_ENVS environments (a reset of the oracle, then edited):
    - BLIND_ENV: the cameras side by side near one corner, at the minimum viewing angle looking into it, the targets and
      obstacles near the opposite corner, out of every camera's range: no camera sees anything but itself;
    - CLUSTER_ENV: every entity within a few units of one point, target 1, camera 0 and obstacle 0 exactly at target 0:
      every target sees every entity, some at relative (0, 0);
    - CORNER_ENVS: target 0 in one terrain corner and the other entities of index 0 and 1 in the opposite one (the second
      environment mirrored), so that relative coordinates reach +-2 terrain sizes;
    - everywhere: the warehouses of TRUE_EMPTY have no cargo left and the others have some, and every target believes
      a different set of empty warehouses."""
    from oracle.oracle import Oracle

    nc, nt, no = cfg['num_cameras'], cfg['num_targets'], cfg['num_obstacles']
    rng = np.random.RandomState(seed)
    oracle = Oracle(cfg, EDGE_ENVS)
    oracle.reset(seed=seed)
    st = oracle.get_state()
    st['episode_step'][:] = 0
    for e in range(EDGE_ENVS):
        for w in range(4):
            st['remaining'][e, w] = 0 if (TRUE_EMPTY[e] >> w) & 1 else np.maximum(st['remaining'][e, w], 1)
        st['tgt_empty_bits'][e] = TRUE_EMPTY[e] ^ (1 + np.arange(nt) % 15)
    # the blind cameras: side by side near one corner, looking into it; everything else near the opposite corner
    st['tgt_xy'][BLIND_ENV] = 850.0 + rng.uniform(-20.0, 20.0, (nt, 2))
    st['obs_xyr'][BLIND_ENV, :, :2] = 850.0 + rng.uniform(-20.0, 20.0, (no, 2))
    side = 60.0 * (np.arange(nc) - (nc - 1) / 2) / np.sqrt(2.0)
    st['cam_xy'][BLIND_ENV] = -800.0 + np.stack([side, -side], axis=-1)
    st['cam_phi'][BLIND_ENV] = -135.0
    st['cam_theta'][BLIND_ENV] = cfg['camera_min_viewing_angle']
    # the cluster
    q = np.array([300.0, -200.0])
    st['tgt_xy'][CLUSTER_ENV] = q + rng.uniform(-5.0, 5.0, (nt, 2))
    st['tgt_xy'][CLUSTER_ENV, 1 % nt] = st['tgt_xy'][CLUSTER_ENV, 0]
    st['cam_xy'][CLUSTER_ENV] = q + rng.uniform(-5.0, 5.0, (nc, 2))
    st['obs_xyr'][CLUSTER_ENV, :, :2] = q + rng.uniform(-5.0, 5.0, (no, 2))
    if nc:
        st['cam_xy'][CLUSTER_ENV, 0] = st['tgt_xy'][CLUSTER_ENV, 0]
    if no:
        st['obs_xyr'][CLUSTER_ENV, 0, :2] = st['tgt_xy'][CLUSTER_ENV, 0]
    # opposite corners
    for e, sign in zip(CORNER_ENVS, (1.0, -1.0)):
        far = sign * np.array([1000.0, 1000.0])
        st['tgt_xy'][e, 0] = -far
        st['tgt_xy'][e, 1:2] = far
        st['cam_xy'][e, :2] = far
        st['obs_xyr'][e, :2, :2] = far
    oracle.set_state(st)
    return oracle.get_state()


def batch_states(cfg):
    """One ragged batch: ORACLE_ENVS reset states of the oracle at staggered episode steps (the next steps auto-reset some
    of them), then the edge batch."""
    from oracle.oracle import Oracle

    oracle = Oracle(cfg, ORACLE_ENVS)
    oracle.reset(seed=SEED)
    st = oracle.get_state()
    st['episode_step'] = np.random.RandomState(SEED).randint(0, LIMIT, ORACLE_ENVS).astype(np.int32)
    edge = edge_states(cfg)
    return {k: np.concatenate([st[k], edge[k]]) for k in st}


@pytest.mark.parametrize('shape', SHAPES, ids=_ids(SHAPES))
def test_edge_batch_holds_its_cases(shape):
    """CPU: the oracle's view of the edge batch has what the GPU tests rely on."""
    from oracle.oracle import Oracle

    nc, nt, no = shape
    cfg = _flat(shape)
    st = edge_states(cfg)
    oracle = Oracle(cfg, EDGE_ENVS)
    oracle.set_state(st)
    aux = oracle.alloc_aux()
    oracle.observe(aux=aux)
    if nc:
        assert not aux['mask_ct'][BLIND_ENV].any() and not aux['mask_co'][BLIND_ENV].any()
        assert np.array_equal(aux['mask_cc'][BLIND_ENV], np.eye(nc, dtype=aux['mask_cc'].dtype))
    for key in ('mask_tc', 'mask_to', 'mask_tt'):
        assert aux[key][CLUSTER_ENV].all(), key
    at0 = st['tgt_xy'][CLUSTER_ENV, 0]
    assert nt == 1 or np.array_equal(st['tgt_xy'][CLUSTER_ENV, 1], at0)
    assert not nc or np.array_equal(st['cam_xy'][CLUSTER_ENV, 0], at0)
    assert not no or np.array_equal(st['obs_xyr'][CLUSTER_ENV, 0, :2], at0)
    for e in CORNER_ENVS:
        others = [st['tgt_xy'][e, 1:2], st['cam_xy'][e, :2], st['obs_xyr'][e, :2, :2]]
        gap = np.concatenate([o.reshape(-1, 2) for o in others]) - st['tgt_xy'][e, 0]
        assert len(gap) and (np.abs(gap) == 2000.0).all()
    truth = (st['remaining'].sum(axis=-1) == 0) @ (1 << np.arange(4))
    assert list(truth) == list(TRUE_EMPTY)
    assert (st['tgt_empty_bits'] != truth[:, None]).all()


# --------------------------------------------------------------------------------------------------- comparisons (GPU)
def _want(ops, raw, state, shape, tables=None):
    """(restated rows, rows before RescaledObservation or None) of the stack `ops` from the raw rows of a point."""
    cam, tgt = raw
    if ops and ops[-1] == RESC:
        x = ref.apply_ops(ops[:-1], cam, tgt, state, shape)
        return ref.apply_ops([RESC], *x, state, shape, tables=tables), x
    return ref.apply_ops(ops, cam, tgt, state, shape), None


def _compare(got, want, before, tables, ctx):
    """Rows of the library (float32, [B, N, D] per team) against the restatement: bit for bit after rounding it to float32,
    or, after RescaledObservation, |k - r| <= 2^-22 (|x s| + |sh| + |r|) with x the value before rescaling and (s, sh)
    the float32 (scale, shift) of the column."""
    for team in range(2):
        k, r = got[team], want[team]
        if k is None or k.size == 0:
            continue
        if before is None:
            bad = k != r.astype(np.float32)
            tol = None
        else:
            s, sh = (np.asarray(tables[team], dtype=np.float64)[:, j] for j in range(2))
            tol = 2.0 ** -22 * (np.abs(before[team] * s) + np.abs(sh) + np.abs(r))
            bad = ~(np.abs(k.astype(np.float64) - r) <= tol)
        if bad.any():
            b, n, d = np.argwhere(bad)[0]
            detail = f'got {k[b, n, d]!r} want {r[b, n, d]!r}' + ('' if before is None else f' x {before[team][b, n, d]!r}')
            raise AssertionError(f'{ctx} {("camera", "target")[team]} rows: {int(bad.sum())} entries differ, first env {b} '
                                 f'row {n} column {d}: {detail}')


def _bits(t):
    import torch

    return t.view(torch.int16 if t.dtype == torch.float16 else torch.int32)


def _same_bits(a, b):
    import torch

    return a is None or b is None or torch.equal(_bits(a), _bits(b))


def _host(rows):
    return tuple(None if t is None else t.cpu().numpy() for t in rows)


def _actions(cfg, B):
    import torch

    rng = np.random.RandomState(SEED + 1)
    nc, nt = cfg['num_cameras'], cfg['num_targets']
    out = []
    for _ in range(STEPS):
        cam = rng.uniform(-1, 1, (B, nc, 2)) * [cfg['camera_rotation_step'], cfg['camera_zooming_step']] if nc else np.zeros((B, 0, 2))
        tgt = rng.uniform(-1, 1, (B, nt, 2)) * cfg['target_step_size']
        out.append((torch.from_numpy(cam.astype(np.float32)).cuda(), torch.from_numpy(tgt.astype(np.float32)).cuda()))
    return out


def _points(sim, states, actions):
    """The rows of `sim` after set_state + observe() and after every step(auto_reset=True) of `actions`."""
    sim.set_state(states)
    yield sim.observe()
    for cam, tgt in actions:
        rows, _, _ = sim.step(cam, tgt, auto_reset=True)
        yield rows


def _twin_points(cfg, states, actions):
    """Raw rows (host) and state of a simulator without wrappers at every point."""
    from mate_b200.sim import BatchedSim

    B = len(states['episode_step'])
    twin = BatchedSim(cfg, B, device=0)
    twin.seed(SEED)
    out, resets = [], []
    for rows in _points(twin, states, actions):
        out.append((_host(rows), twin.get_state()))
        resets.append(int(twin.done.sum()) if len(out) > 1 else 0)
    assert 0 < max(resets) < B and all(r < B for r in resets), resets   # some environments were auto-reset
    twin.close()
    return out


def _register(sim, ops, monkeypatch, fold=True):
    if fold:
        monkeypatch.delenv('MATE_B200_FOLD', raising=False)
    else:
        monkeypatch.setenv('MATE_B200_FOLD', '0')   # read when the ops are set
    sim.set_observation_wrappers(ops)
    monkeypatch.delenv('MATE_B200_FOLD', raising=False)


@pytest.mark.gpu
@pytest.mark.parametrize('shape', SHAPES, ids=_ids(SHAPES))
def test_every_stack_on_every_path(shape, monkeypatch):
    """GPU, every stack of STACKS on oracle states (ragged batch, steps with auto-resets) and the edge batch:
    - the folded fast path and the generic path against the restatement (bit for bit, or within the rescale bound);
    - the fast path, the generic path and the separate pass bit-identical;
    - float16 rows = the float32 rows rounded to nearest even, bit for bit;
    - single-team rows = the matching rows of the both-teams simulator (stacks with RelativeCoordinates or
      RescaledObservation);
    - caller tables that differ between two targets' entries: the generic path, equal to the restatement with those tables."""
    import torch

    from mate_b200.sim import BatchedSim, rescale_tables

    nc, nt, no = shape
    monkeypatch.delenv('MATE_B200_FOLD', raising=False)
    cfg = _flat(shape, max_episode_steps=LIMIT)
    states = batch_states(cfg)
    B = len(states['episode_step'])
    actions = _actions(cfg, B)
    points = _twin_points(cfg, states, actions)
    tables = rescale_tables(nc, nt, no)

    def make(**kw):
        sim = BatchedSim(cfg, B, device=0, **kw)
        sim.seed(SEED)
        return sim

    fast, generic, sep, half = make(), make(), make(), make(observation_dtype=torch.float16)
    singles = [make(observed_team=team) for team in (('camera', 'target') if nc else ('target',))]
    for ops in STACKS:
        _register(fast, ops, monkeypatch)
        _register(generic, ops, monkeypatch, fold=False)
        _register(half, ops, monkeypatch)
        tail = REL in ops or RESC in ops
        sims = [fast, generic, sep, half] + (singles if tail else [])
        for single in singles if tail else []:
            _register(single, ops, monkeypatch)
        for k, rows in enumerate(zip(*(_points(sim, states, actions) for sim in sims))):
            ctx = f'{preset_of(shape)} [{_name(ops)}] point {k}'
            raw, state = points[k]
            want, before = _want(ops, raw, state, shape)
            a, g = rows[0], rows[1]
            _compare(_host(a), want, before, tables, ctx + ' fast path')
            _compare(_host(g), want, before, tables, ctx + ' generic path')
            assert _same_bits(a[0], g[0]) and _same_bits(a[1], g[1]), ctx + ' fast vs generic'
            sep.set_observation_wrappers(ops)
            sep.transform_observations()      # the separate pass over the raw rows
            assert _same_bits(a[0], rows[2][0]) and _same_bits(a[1], rows[2][1]), ctx + ' fast vs separate pass'
            sep.set_observation_wrappers([])
            h = rows[3]
            assert _same_bits(h[0], None if a[0] is None else a[0].half()) and _same_bits(h[1], a[1].half()), ctx + ' float16'
            for single, one in zip(singles if tail else [], rows[4:]):
                team = 0 if single.observed_team == 'camera' else 1
                assert one[1 - team] is None and _same_bits(one[team], a[team]), ctx + f' {single.observed_team} rows only'

    # caller tables that are not uniform per kind: the library has to take the generic path
    if nt > 1:
        custom = make()
        skewed = (tables[0], _skew(tables[1], shape))
        dev = [torch.from_numpy(t).cuda() for t in skewed]
        for ops in ((RESC,), (SH_C, SH_T, REL, RESC)):
            codes = (ctypes.c_int32 * len(ops))(*ops)
            with torch.cuda.device(custom.device):
                rc = custom.lib.mate_b200_set_observation_ops(custom.handle, codes, len(ops),
                                                              ctypes.c_void_p(dev[0].data_ptr()) if nc else None,
                                                              ctypes.c_void_p(dev[1].data_ptr()))
            assert rc == 0, custom.lib.mate_b200_last_error()
            for k, rows in enumerate(_points(custom, states, actions)):
                raw, state = points[k]
                want, before = _want(ops, raw, state, shape, tables=skewed)
                _compare(_host(rows), want, before, skewed, f'{preset_of(shape)} [{_name(ops)}] point {k} skewed tables')
        custom.close()
    for sim in [fast, generic, sep, half] + singles:
        sim.close()


TILE_SHAPES = [(0, 8, 32), (1, 2, 9), (2, 2, 9), (8, 8, 9)]


@pytest.mark.gpu
@pytest.mark.parametrize('shape', TILE_SHAPES, ids=_ids(TILE_SHAPES))
def test_rescaled_stacks_in_every_warp_tile(shape, monkeypatch):
    """GPU: the stacks with RescaledObservation on the fast path in warp tiles of 8, 16 and 32 environments (the
    rescaled constants are staged once per tile; the batch leaves the last tile partial) against the restatement."""
    from mate_b200.sim import BatchedSim, rescale_tables

    monkeypatch.delenv('MATE_B200_FOLD', raising=False)
    cfg = _flat(shape, max_episode_steps=LIMIT)
    states = batch_states(cfg)
    B = len(states['episode_step'])
    assert B % 32 and B % 16 and B % 8
    actions = _actions(cfg, B)
    points = _twin_points(cfg, states, actions)
    tables = rescale_tables(*shape)
    sims = []
    for tile in ('8', '16', '32'):
        monkeypatch.setenv('MATE_B200_TILE', tile)   # read when the simulator is created
        sims.append(BatchedSim(cfg, B, device=0))
        sims[-1].seed(SEED)
    monkeypatch.delenv('MATE_B200_TILE')
    for ops in [s for s in STACKS if RESC in s]:
        for sim in sims:
            sim.set_observation_wrappers(ops)
        for k, rows in enumerate(zip(*(_points(sim, states, actions) for sim in sims))):
            raw, state = points[k]
            want, before = _want(ops, raw, state, shape)
            for tile, got in zip((8, 16, 32), rows):
                _compare(_host(got), want, before, tables, f'{preset_of(shape)} [{_name(ops)}] point {k} tile {tile}')
    for sim in sims:
        sim.close()


@pytest.mark.gpu
@pytest.mark.parametrize('shape', [(4, 8, 9), (0, 8, 32)], ids=_ids([(4, 8, 9), (0, 8, 32)]))
def test_refused_orders_leave_the_registered_stack(shape):
    """GPU: every forbidden order is refused by set_observation_wrappers (ValueError) and, through the C ABI, by
    mate_b200_set_observation_ops and mate_b200_transform_observations (MATE_EINVAL); the stack registered before
    stays in effect."""
    import torch

    from mate_b200.sim import BatchedSim

    cfg = _flat(shape)
    sim = BatchedSim(cfg, 37, device=0)
    sim.reset(seed=4)
    sim.set_observation_wrappers([SH_C, SH_T, REL, RESC])
    before = [t.clone() for t in sim.observe() if t is not None]
    cam_aff, tgt_aff = sim._affine   # pylint: disable=protected-access
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for ops in FORBIDDEN:
        with pytest.raises(ValueError):
            sim.set_observation_wrappers(ops)
        codes = (ctypes.c_int32 * len(ops))(*ops)
        aff = (ctypes.c_void_p(cam_aff.data_ptr()) if sim.nc else None, ctypes.c_void_p(tgt_aff.data_ptr()))
        with torch.cuda.device(sim.device):
            assert sim.lib.mate_b200_set_observation_ops(sim.handle, codes, len(ops), *aff) == -1, ops
            scratch = [torch.zeros_like(t) if t is not None else None for t in (sim.cam_obs, sim.tgt_obs)]
            ptrs = [ctypes.c_void_p(t.data_ptr()) if t is not None else None for t in scratch]
            assert sim.lib.mate_b200_transform_observations(sim.handle, *ptrs, codes, len(ops), *aff, stream) == -1, ops
        assert b'Relative? Rescaled?' in sim.lib.mate_b200_last_error()
        assert all(t is None or not t.any() for t in scratch)
        after = [t for t in sim.observe() if t is not None]
        assert all(torch.equal(_bits(x), _bits(y)) for x, y in zip(before, after)), ops
    assert sim._obs_ops == [SH_C, SH_T, REL, RESC]   # pylint: disable=protected-access
    sim.close()
