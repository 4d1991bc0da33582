"""NumPy float64 restatement of the reference's observation wrappers -- TEST INFRASTRUCTURE: the checker of the
wrapper code of the step kernel's packer and of ``mate_b200_transform_observations``, itself pinned against the
reference's values in ``tests/golden/wrappers_*.npz``.  Restated behaviour (reference root):
  EnhancedObservation.observation   mate/wrappers/enhanced_observation.py:72-123
  SharedFieldOfView.observation     mate/wrappers/shared_field_of_view.py:74-145
  convert_coordinates               mate/agents/utils.py:40-94   (RelativeCoordinates)
  normalize_observation             mate/agents/utils.py:97-127  (RescaledObservation)

It works from raw observation rows ``[B, N, D]`` and the state (``tgt_xy``, ``cam_xy``, ``obs_xyr``, ``remaining``), is
vectorised over the batch and loops over entities only.  From ``mate_b200`` it uses the layout constants and observation
spaces of ``mate_b200/constants.py`` and nothing else (in particular not the library's float32 rescale tables)."""

import numpy as np

from mate_b200 import constants as C

# wrapper codes, innermost first (MATE_OBS_* of include/mate_b200.h)
ENHANCED_CAMERA, ENHANCED_TARGET, SHARED_CAMERA, SHARED_TARGET, RELATIVE, RESCALED = range(1, 7)
MASK_OPS = (ENHANCED_CAMERA, ENHANCED_TARGET, SHARED_CAMERA, SHARED_TARGET)
P, NW = C.PRESERVED_DIM, C.NUM_WAREHOUSES
EMPTY = P + C.TARGET_STATE_DIM_PRIVATE - NW            # first empty bit of a target row
WIDTH = {'tgt': C.TARGET_STATE_DIM_PUBLIC, 'obs': C.OBSTACLE_STATE_DIM, 'cam': C.CAMERA_STATE_DIM_PUBLIC}


def blocks(team, shape):
    """(kind, public width, count, first column) of the opponent, obstacle and teammate blocks of a `team` row."""
    nc, nt, no = shape
    idx = C.observation_indices_of(team, nc, nt, no)
    kinds = ('tgt', 'obs', 'cam') if team == 'camera' else ('cam', 'obs', 'tgt')
    counts = {'tgt': nt, 'obs': no, 'cam': nc}
    return [(k, WIDTH[k], counts[k], int(idx[2 + i])) for i, k in enumerate(kinds)]


def _public(cam, tgt, state, shape):
    """Public states [B, n, w] by kind: cameras and targets from the own-row blocks of the rows, obstacles from the state."""
    nc, _, no = shape
    return {'cam': cam[:, :, P:P + WIDTH['cam']], 'tgt': tgt[:, :, P:P + WIDTH['tgt']],
            'obs': np.asarray(state['obs_xyr'], dtype=np.float64)[:, :no]}


def _mask_op(op, rows, cam, tgt, state, shape):
    team = 'camera' if op in (ENHANCED_CAMERA, SHARED_CAMERA) else 'target'
    R = rows[team]
    if R.shape[1] == 0:               # no cameras: the camera team's wrappers do nothing
        return
    shared = op in (SHARED_CAMERA, SHARED_TARGET)
    pub = _public(cam, tgt, state, shape)
    own = 'cam' if team == 'camera' else 'tgt'
    for kind, w, n, first in blocks(team, shape):
        for e in range(n):
            o = first + (w + 1) * e
            slot = np.append(pub[kind][:, e], np.ones((R.shape[0], 1)), axis=-1)[:, None, :]   # [B, 1, w + 1]
            if shared:   # teammates always; another entity iff some member of the team sees it
                seen = np.full(R.shape[0], True) if kind == own else (R[:, :, o + w] != 0).any(axis=1)
                slot = np.where(seen[:, None, None], slot, 0.0)
            R[:, :, o:o + w + 1] = slot
    if team == 'target':
        if shared:   # the team's beliefs, "or"-ed
            bits = (R[:, :, EMPTY:EMPTY + NW] != 0).any(axis=1)
        else:        # the truth: no cargo left at the warehouse
            bits = np.asarray(state['remaining']).sum(axis=-1) == 0
        R[:, :, EMPTY:EMPTY + NW] = bits[:, None, :].astype(np.float64)


def _relative(rows, state, shape):
    nc, nt, no = shape
    loc = {'tgt': np.asarray(state['tgt_xy'], dtype=np.float64)[:, :nt],
           'obs': np.asarray(state['obs_xyr'], dtype=np.float64)[:, :no, :2],
           'cam': np.asarray(state['cam_xy'], dtype=np.float64)[:, :nc]}
    for team, R in rows.items():
        own = loc['cam' if team == 'camera' else 'tgt']                 # [B, N, 2]; the own location stays absolute
        R[:, :, 4:4 + 2 * NW] -= np.tile(own, NW)                        # the warehouses
        for kind, w, n, first in blocks(team, shape):
            for e in range(n):
                o = first + (w + 1) * e
                flagged = (R[:, :, o + w] != 0)[..., None]
                R[:, :, o:o + 2] = np.where(flagged, loc[kind][:, e][:, None, :] - own, R[:, :, o:o + 2])


def normalize(x, space):
    """normalize_observation in float64 from the space bounds: columns bounded on both sides to [-1, 1], columns bounded
    below only shifted by their lower bound, the others unchanged.  The reference's (x - low) * 2 / (high - low) - 1 is
    evaluated as x * scale + shift with float64 (scale, shift): the same map, without the cancellation of x - low, so
    that an entry close to zero keeps its relative precision (the two forms differ by ~1e-16)."""
    low, high = np.asarray(space.low, dtype=np.float64), np.asarray(space.high, dtype=np.float64)
    both, below = np.isfinite(low) & np.isfinite(high), np.isfinite(low) & ~np.isfinite(high)
    scale = 2.0 / (high[both] - low[both])
    out = x.copy()
    out[..., both] = x[..., both] * scale + (-low[both] * scale - 1.0)
    out[..., below] = x[..., below] - low[below]
    return out


def apply_ops(ops, cam_rows, tgt_rows, state, shape, tables=None):
    """The wrapper codes `ops` (innermost first) applied to raw rows ``cam_rows [B, Nc, Dc]`` / ``tgt_rows [B, Nt, Dt]`` of
    the state `state`; returns float64 ``(cam, tgt)``.  `tables` = ``(cam_table [Dc, 2], tgt_table [Dt, 2])`` replaces
    normalize_observation with ``x * scale + shift`` from the caller's (scale, shift) columns."""
    nc, nt, no = shape
    cam, tgt = np.array(cam_rows, dtype=np.float64), np.array(tgt_rows, dtype=np.float64)
    rows = {'camera': cam, 'target': tgt}
    for op in ops:
        if op in MASK_OPS:
            _mask_op(op, rows, cam, tgt, state, shape)
        elif op == RELATIVE:
            _relative(rows, state, shape)
        elif op == RESCALED:
            for team, R in rows.items():
                if tables is not None:
                    t = np.asarray(tables[0 if team == 'camera' else 1], dtype=np.float64)
                    R[...] = R * t[:, 0] + t[:, 1]
                else:
                    R[...] = normalize(R, C.observation_space_of(team, nc, nt, no))
        else:
            raise ValueError(f'unknown observation wrapper code {op}')
    return cam, tgt
