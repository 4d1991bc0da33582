"""Low-level Python binding of the C ABI (``include/mate_b200.h``).

PyTorch is used only for device memory and streams: tensors are allocated here and their
raw device pointers are handed to ``libmate_b200.so``.  There is no CPU path.
"""

import ctypes

import numpy as np
import torch

from mate_b200 import _abi


class MateError(RuntimeError):
    pass


def _check(lib, rc):
    if rc != 0:
        msg = lib.mate_b200_last_error().decode('utf-8', 'replace')
        if rc == -1:
            raise ValueError(msg)
        raise MateError(f'mate_b200 error {rc}: {msg}')


def _dptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def rescale_tables(nc, nt, no):
    """(scale, shift) per observation column so that ``x * scale + shift`` equals the reference's
    ``normalize_observation`` (mate/agents/utils.py:97-127): subtract ``low`` where it is finite, then map the
    columns that are bounded on both sides (and not degenerate) to [-1, 1].  float32 [D][2] per team."""
    from mate_b200 import constants as consts  # pylint: disable=import-outside-toplevel

    tables = []
    for space in (consts.camera_observation_space_of(nc, nt, no), consts.target_observation_space_of(nc, nt, no)):
        low, high = np.asarray(space.low, dtype=np.float64), np.asarray(space.high, dtype=np.float64)
        below, above = np.isfinite(low), np.isfinite(high)
        both = below & above & (np.where(below & above, high - low, 0.0) > 0.0)
        span = np.where(both, high - low, 1.0)
        scale = np.where(both, 2.0 / span, 1.0)
        shift = np.where(below, -low, 0.0) * scale + np.where(both, -1.0, 0.0)
        tables.append(np.stack([scale, shift], axis=-1).astype(np.float32))
    return tuple(tables)


OBSERVATION_FORMATS = {torch.float32: _abi.MATE_OBS_FORMAT_F32, torch.float16: _abi.MATE_OBS_FORMAT_F16}


def check_observation_dtype(dtype):
    """The element type of the observation rows: ``torch.float32`` or ``torch.float16`` (rounded once, to nearest even,
    from the float32 rows), else ``ValueError``."""
    if dtype not in OBSERVATION_FORMATS:
        raise ValueError(f'observation_dtype must be torch.float32 or torch.float16, got {dtype!r}')
    return dtype


def check_observation_ops(ops):
    """Observation wrapper codes (``_abi.OBS_*``) as a list of ints, else ``ValueError``: at most ``MAX_OBS_OPS`` known
    codes in the order the reference's wrappers admit, ``(Enhanced | Shared)* Relative? Rescaled?`` (no mask code after
    ``OBS_RELATIVE`` or ``OBS_RESCALED``, neither of those twice, no ``OBS_RELATIVE`` after ``OBS_RESCALED``)."""
    ops = [int(op) for op in ops]
    if len(ops) > _abi.MAX_OBS_OPS:
        raise ValueError(f'at most {_abi.MAX_OBS_OPS} observation wrappers can be stacked')
    stage = 0   # 0 = mask codes, 1 = after OBS_RELATIVE, 2 = after OBS_RESCALED
    for op in ops:
        if not _abi.OBS_ENHANCED_CAMERA <= op <= _abi.OBS_RESCALED:
            raise ValueError(f'unknown observation wrapper code {op}')
        at = {_abi.OBS_RELATIVE: 1, _abi.OBS_RESCALED: 2}.get(op, 0)
        if at < stage or (at > 0 and at == stage):
            raise ValueError(f'observation wrappers must be stacked as (Enhanced | Shared)* Relative? Rescaled?, got {ops}')
        stage = at
    return ops


OBSERVED_TEAMS = ('both', 'camera', 'target')


def check_observed_team(team, num_cameras=None):
    """Whose observation rows a batched simulator composes and writes: ``'both'``, ``'camera'`` or ``'target'``, else
    ``ValueError``; ``'camera'`` also needs cameras (``num_cameras``, when given)."""
    if not isinstance(team, str) or team not in OBSERVED_TEAMS:
        raise ValueError(f'observed_team must be one of {OBSERVED_TEAMS}, got {team!r}')
    if team == 'camera' and num_cameras == 0:
        raise ValueError("observed_team='camera' needs a configuration with cameras")
    return team


def check_index_map(index, name, length, low, high):
    """The checks of an environment / snapshot index map, before any library call: 1-D integers, ``length`` of them if
    given, and for a host sequence (or CPU tensor) each in ``[low, high)``, else ``ValueError``.  Returns the host indices
    as a NumPy array, or ``None`` for ``None`` and for a device tensor (its entries are not read here)."""
    if index is None:
        return None
    if torch.is_tensor(index) and index.is_cuda:
        if index.dtype.is_floating_point or index.dtype.is_complex or index.dtype == torch.bool:
            raise ValueError(f'{name} must hold integers, got {index.dtype}')
        host = None
    else:
        host = index.numpy() if torch.is_tensor(index) else np.asarray(index)
        if host.dtype.kind not in 'iu':
            raise ValueError(f'{name} must hold integers, got {host.dtype}')
    size = tuple(index.shape) if host is None else host.shape
    if len(size) != 1 or size[0] == 0 or (length is not None and size[0] != length):
        raise ValueError(f'{name} must be a 1-D sequence of {length if length is not None else "one or more"} indices, got shape {size}')
    if host is not None and (host.min() < low or host.max() >= high):
        raise ValueError(f'{name} has entries outside [{low}, {high})')
    return host


def check_render_size(size):
    """The edge of a rendered frame in pixels: an integer in ``[MATE_RENDER_MIN_SIZE, MATE_RENDER_MAX_SIZE]``, else
    ``ValueError``."""
    if isinstance(size, bool) or not isinstance(size, (int, np.integer)) or not _abi.RENDER_MIN_SIZE <= size <= _abi.RENDER_MAX_SIZE:
        raise ValueError(f'the frame size must be an integer in [{_abi.RENDER_MIN_SIZE}, {_abi.RENDER_MAX_SIZE}], got {size!r}')
    return int(size)


class StateSnapshot:
    """The complete state of some environments of a batch, saved on the device (:meth:`BatchedSim.save_state`).

    ``payload`` is a ``uint8`` tensor in the library's private layout; the header fields are those of
    ``MateSnapshotInfo`` (``include/mate_b200.h``); ``py_seed`` is the saving simulator's Python-side seed, and
    ``extras`` holds the per-snapshot state of the Python layers above the simulator (environment RNG, opponent
    agents).  ``torch.save`` / ``torch.load`` keep it as it is; a payload on the CPU or on another GPU is copied to the
    loading simulator's device."""

    def __init__(self, payload, py_seed=0, extras=None, **header):
        self.payload = payload
        for name in _abi.SNAPSHOT_INFO_FIELDS:
            setattr(self, name, int(header[name]))
        self.py_seed = int(py_seed)
        self.extras = {} if extras is None else extras

    def info(self):
        """The header as a ``MateSnapshotInfo``."""
        return _abi.MateSnapshotInfo(**{name: getattr(self, name) for name in _abi.SNAPSHOT_INFO_FIELDS})

    def __repr__(self):
        return (f'StateSnapshot(count={self.count}, shape=({self.num_cameras}, {self.num_targets}, {self.num_obstacles}), '
                f'{self.payload_bytes} bytes on {self.payload.device})')


torch.serialization.add_safe_globals([StateSnapshot])   # torch.load(weights_only=True), the default, accepts it


class BatchedSim:
    """One batch of MultiAgentTracking environments resident on one GPU.  ``observation_dtype`` is the element type of
    the observation rows (``cam_obs`` / ``tgt_obs``); everything else stays float32.  ``observed_team`` (``'both'``,
    ``'camera'`` or ``'target'``) is whose rows are composed and written: the other team's tensor is ``None`` and its
    rows cost nothing; everything else is what a ``'both'`` simulator computes."""

    def __init__(self, flat_config, num_envs, device=0, env_index_base=0, observation_dtype=torch.float32, observed_team='both'):
        self.observation_dtype = check_observation_dtype(observation_dtype)
        self.observed_team = check_observed_team(observed_team, int(dict(flat_config)['num_cameras']))
        if not torch.cuda.is_available():
            raise RuntimeError('mate_b200 needs a CUDA device (there is no CPU fallback)')
        self.lib = _abi.load_library()
        self.cfg = dict(flat_config)
        self._cfg_struct = _abi.make_config_struct(self.cfg)
        self.B = int(num_envs)
        self.nc = int(self.cfg['num_cameras'])
        self.nt = int(self.cfg['num_targets'])
        self.no = int(self.cfg['num_obstacles'])
        index = device if isinstance(device, int) else (torch.device(device).index or 0)
        self.device = torch.device('cuda', index)
        self.handle = ctypes.c_void_p()
        _check(self.lib, self.lib.mate_b200_create(ctypes.byref(self._cfg_struct), self.B, self.device.index,
                                                   int(env_index_base), ctypes.byref(self.handle)))
        _check(self.lib, self.lib.mate_b200_set_observation_format(self.handle, OBSERVATION_FORMATS[self.observation_dtype]))
        dc, dt = ctypes.c_int32(), ctypes.c_int32()
        _check(self.lib, self.lib.mate_b200_obs_dims(self.handle, ctypes.byref(dc), ctypes.byref(dt)))
        self.dc, self.dt = dc.value, dt.value
        dev = self.device
        self.cam_obs, self.tgt_obs = (
            torch.zeros(shape, dtype=self.observation_dtype, device=dev) if self.observed_team in ('both', team) else None
            for team, shape in (('camera', (self.B, self.nc, self.dc)), ('target', (self.B, self.nt, self.dt))))
        self.rewards = torch.zeros((self.B, 2), dtype=torch.float32, device=dev)
        self.done = torch.zeros((self.B,), dtype=torch.uint8, device=dev)
        self._stats = torch.zeros(16, dtype=torch.float32, device=dev)
        self._aux = None
        self._aux_struct = None
        self._zero_cam_act = torch.zeros((self.B, max(self.nc, 1), 2), dtype=torch.float32, device=dev)
        self._obs_ops, self._obs_ops_c, self._affine = [], None, None
        self._seed = 0

    def close(self):
        if getattr(self, 'handle', None) is not None and self.handle:
            self.lib.mate_b200_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # pylint: disable=broad-except
            pass

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def alloc_aux(self):
        """Device tensors for every MateStepAux field."""
        tmap = {np.uint8: torch.uint8, np.float32: torch.float32, np.int32: torch.int32}
        self._aux = {
            name: torch.zeros(shape(self.B, self.nc, self.nt, self.no), dtype=tmap[dtype], device=self.device)
            for name, _, dtype, shape in _abi.AUX_FIELDS
        }
        s = _abi.MateStepAux()
        for name, ctype, _, _ in _abi.AUX_FIELDS:
            setattr(s, name, ctypes.cast(ctypes.c_void_p(self._aux[name].data_ptr()), ctype))
        self._aux_struct = s
        return self._aux

    @property
    def aux(self):
        if self._aux is None:
            self.alloc_aux()
        return self._aux

    def _replay_struct(self, replay):
        if replay is None:
            return None, None
        transmit, choice = replay
        keep = []
        s = _abi.MateReplay()
        if transmit is not None:
            t = torch.as_tensor(np.ascontiguousarray(transmit, dtype=np.uint8)).to(self.device)
            t = t.reshape(self.B, self.nc, self.nt).contiguous()
            keep.append(t)
            s.transmit = ctypes.cast(ctypes.c_void_p(t.data_ptr()), _abi.c_uint8_p)
        if choice is not None:
            c = torch.as_tensor(np.ascontiguousarray(choice, dtype=np.int8)).to(self.device)
            c = c.reshape(self.B, self.nt).contiguous()
            keep.append(c)
            s.goal_choice = ctypes.cast(ctypes.c_void_p(c.data_ptr()), _abi.c_int8_p)
        return s, keep

    def _actions(self, cam_act, tgt_act):
        tgt_act = torch.as_tensor(tgt_act, dtype=torch.float32, device=self.device)
        tgt_act = tgt_act.reshape(self.B, self.nt, 2).contiguous()
        if self.nc:
            cam_act = torch.as_tensor(cam_act, dtype=torch.float32, device=self.device)
            cam_act = cam_act.reshape(self.B, self.nc, 2).contiguous()
        else:
            cam_act = self._zero_cam_act
        return cam_act, tgt_act

    # ------------------------------------------------------------------ observation wrappers (N1)
    def set_observation_wrappers(self, ops):
        """Observation wrapper codes (``_abi.OBS_*``), innermost first.  They are registered with the simulator
        (``mate_b200_set_observation_ops``): every reset / step / observe applies them to an environment's rows while
        the rows are still in shared memory, at no extra pass over the observation tensors."""
        ops = check_observation_ops(ops)
        self._obs_ops = ops
        self._obs_ops_c = (ctypes.c_int32 * max(len(ops), 1))(*ops)
        if _abi.OBS_RESCALED in ops and self._affine is None:
            self._affine = tuple(torch.from_numpy(t).to(self.device) for t in rescale_tables(self.nc, self.nt, self.no))
        cam_aff, tgt_aff = self._affine if self._affine is not None else (None, None)
        _check(self.lib, self.lib.mate_b200_set_observation_ops(
            self.handle, self._obs_ops_c, len(ops), _dptr(cam_aff) if (self.nc and cam_aff is not None) else None, _dptr(tgt_aff)))

    def transform_observations(self):
        """The registered wrappers as a separate in-place pass over the current observation tensors
        (``mate_b200_transform_observations``); only for tensors that did NOT come out of reset / step / observe with
        the wrappers registered (those are transformed already)."""
        if not self._obs_ops:
            return
        if self.tgt_obs is None or (self.nc and self.cam_obs is None):
            raise ValueError(f"transform_observations needs both teams' rows; this simulator observes {self.observed_team!r} only "
                             '(register the wrappers with set_observation_wrappers instead)')
        cam_aff, tgt_aff = self._affine if self._affine is not None else (None, None)
        with torch.cuda.device(self.device):
            _check(self.lib, self.lib.mate_b200_transform_observations(
                self.handle, _dptr(self.cam_obs), _dptr(self.tgt_obs), self._obs_ops_c, len(self._obs_ops),
                _dptr(cam_aff) if self.nc else None, _dptr(tgt_aff), self._stream()))

    def decode_actions(self, index, table):
        """DiscreteCamera / DiscreteTarget: int64 grid indices [B, N] -> float32 actions [B, N, 2]."""
        index = torch.as_tensor(index, device=self.device).to(torch.int64).contiguous()
        out = torch.empty(tuple(index.shape) + (2,), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _check(self.lib, self.lib.mate_b200_decode_actions(_dptr(index), _dptr(table), int(table.shape[0]), _dptr(out),
                                                               index.numel(), self._stream()))
        return out

    def set_message_filter(self, range_limit=(np.inf, np.inf), keep_probability=(1.0, 1.0), delivered=(None, None),
                           total_edges=(None, None)):
        """Register the communication wrappers with the simulator (mate_b200_set_message_filter): per team (cameras,
        targets) the range limit and the keep probability the batched greedy teams apply to their messages, and the
        device tensors their kernels write the delivered sets to (int64 ``[B]``, bit ``8 s + r``) and add them to
        (int32 ``[B, N, N]``); ``None`` = not counted.  The defaults deliver everything."""
        tensors = []
        for team, n in enumerate((self.nc, self.nt)):
            for name, t, dtype, shape in (('delivered', delivered[team], torch.int64, (self.B,)),
                                          ('total_edges', total_edges[team], torch.int32, (self.B, n, n))):
                if t is not None and (t.device != self.device or t.dtype != dtype or tuple(t.shape) != shape or not t.is_contiguous()):
                    raise ValueError(f'{name}[{team}] must be a contiguous {dtype} tensor of shape {shape} on {self.device}')
                tensors.append(t)
        f = _abi.MateMessageFilter()
        for team in range(2):
            f.range_limit[team] = float(range_limit[team])
            f.keep_probability[team] = float(keep_probability[team])
            f.delivered[team] = None if delivered[team] is None else delivered[team].data_ptr()
            f.total_edges[team] = None if total_edges[team] is None else total_edges[team].data_ptr()
        _check(self.lib, self.lib.mate_b200_set_message_filter(self.handle, ctypes.byref(f)))
        self._message_tensors = tensors   # the library keeps the pointers

    def exchange_messages(self, team, content, recipients, reduction, serial, episode):
        """The tensor message channel of team 0 (cameras) or 1 (targets) (mate_b200_exchange_messages): ``content``
        float32 ``[B, N, D]``, one message per sender; ``recipients`` bool / uint8 ``[B, N, N]`` sender-major (``None`` =
        broadcast); ``reduction`` ``'none'`` / ``'sum'`` / ``'mean'``; ``serial`` keys the dropout draws; ``episode`` is the
        team's int32 ``[B]`` bookkeeping of the episode its totals belong to.  Returns fresh ``(inbox, delivered)``:
        ``inbox`` float32 ``[B, N(r), N(s), D]`` (``'none'``) or ``[B, N(r), D]``, ``delivered`` bool ``[B, N(r), N(s)]``.
        Every argument is checked here, before any library call; nothing synchronises."""
        if team not in (0, 1):
            raise ValueError(f'team must be 0 (cameras) or 1 (targets), got {team!r}')
        n = (self.nc, self.nt)[team]
        if not 0 < n <= 8:
            raise ValueError(f'the message exchange covers teams of 1 to 8 agents (bit 8 s + r); team {team} has {n}')
        if reduction not in _abi.MESSAGE_REDUCTIONS:
            raise ValueError(f"reduction must be one of {sorted(_abi.MESSAGE_REDUCTIONS)}, got {reduction!r}")

        def check(name, t, dtypes, shape):
            if not torch.is_tensor(t) or t.dtype not in dtypes or t.device != self.device or t.dim() != len(shape) \
                    or any(want is not None and got != want for got, want in zip(t.shape, shape)) or not t.is_contiguous():
                kinds = ' or '.join(str(d) for d in dtypes)
                raise ValueError(f'{name} must be a contiguous {kinds} tensor of shape {tuple("D" if s is None else s for s in shape)} '
                                 f'on {self.device}, got {type(t).__name__} {getattr(t, "dtype", "")} {tuple(getattr(t, "shape", ()))} '
                                 f'on {getattr(t, "device", "")}')

        check('content', content, (torch.float32,), (self.B, n, None))
        dim = int(content.shape[2])
        if dim < 1 or n * n * dim >= 1 << 31:
            raise ValueError(f'content must hold 1 to {((1 << 31) - 1) // (n * n)} floats per message, got {dim}')
        if recipients is not None:
            check('recipients', recipients, (torch.bool, torch.uint8), (self.B, n, n))
        check('episode', episode, (torch.int32,), (self.B,))
        out_shape = (self.B, n, n, dim) if reduction == 'none' else (self.B, n, dim)
        inbox = torch.empty(out_shape, dtype=torch.float32, device=self.device)
        delivered = torch.empty((self.B, n, n), dtype=torch.bool, device=self.device)
        x = _abi.MateMessageExchange(content=content.data_ptr(), recipients=None if recipients is None else recipients.data_ptr(),
                                     inbox=inbox.data_ptr(), delivered=delivered.data_ptr(), episode=episode.data_ptr(),
                                     team=team, dim=dim, reduction=_abi.MESSAGE_REDUCTIONS[reduction], reserved=0)
        with torch.cuda.device(self.device):
            _check(self.lib, self.lib.mate_b200_exchange_messages(self.handle, ctypes.byref(x), int(serial) % (1 << 64), self._stream()))
        return inbox, delivered

    # ------------------------------------------------------------------ API
    def seed(self, seed, env_mask=None):
        """``MultiAgentTracking.seed``: new key for the Philox streams, episode counters rewound (mate_b200_seed), so
        that the following resets are reproducible."""
        mask = None
        if env_mask is not None:
            mask = torch.as_tensor(env_mask, device=self.device).to(torch.uint8).contiguous()
        self._seed = int(seed)
        with torch.cuda.device(self.device):
            _check(self.lib, self.lib.mate_b200_seed(self.handle, _dptr(mask), self._seed, self._stream()))

    def reset(self, seed=None, env_mask=None):
        """Reset the environments of ``env_mask`` (default: all).  With an explicit ``seed`` the reset is reproducible
        (``reset(seed=s)`` twice gives the same states, like the reference); without one it draws the next episodes
        of the current seed."""
        mask = None
        if env_mask is not None:
            mask = torch.as_tensor(env_mask, device=self.device).to(torch.uint8).contiguous()
        if seed is not None:
            self.seed(seed, mask)
        with torch.cuda.device(self.device):
            _check(self.lib, self.lib.mate_b200_reset(self.handle, _dptr(mask), self._seed, _dptr(self.cam_obs),
                                                      _dptr(self.tgt_obs), self._stream()))
        return self.cam_obs, self.tgt_obs

    def step(self, cam_act, tgt_act, auto_reset=True, replay=None, aux=False):
        cam_act, tgt_act = self._actions(cam_act, tgt_act)
        rs, keep = self._replay_struct(replay)
        if aux and self._aux is None:
            self.alloc_aux()
        with torch.cuda.device(self.device):
            _check(self.lib, self.lib.mate_b200_step(
                self.handle, _dptr(cam_act), _dptr(tgt_act), _dptr(self.cam_obs), _dptr(self.tgt_obs),
                _dptr(self.rewards), _dptr(self.done),
                ctypes.byref(self._aux_struct) if aux else None,
                ctypes.byref(rs) if rs is not None else None,
                _abi.MATE_STEP_AUTO_RESET if auto_reset else 0, self._stream()))
        del keep
        return (self.cam_obs, self.tgt_obs), self.rewards, self.done

    def observe(self, replay=None, aux=False):
        rs, keep = self._replay_struct(replay)
        if aux and self._aux is None:
            self.alloc_aux()
        with torch.cuda.device(self.device):
            _check(self.lib, self.lib.mate_b200_observe(
                self.handle, _dptr(self.cam_obs), _dptr(self.tgt_obs),
                ctypes.byref(self._aux_struct) if aux else None,
                ctypes.byref(rs) if rs is not None else None, self._stream()))
        del keep
        return self.cam_obs, self.tgt_obs

    def fov_range(self, env, camera, angle_deg):
        """``Camera.sight_range_at`` (mate/entities.py:507-511) for equally shaped arrays of environment indices,
        camera indices and bearings in degrees; float64 tensor of the same shape."""
        env = torch.as_tensor(env, device=self.device).to(torch.int32).contiguous()
        camera = torch.as_tensor(camera, device=self.device).to(torch.int32).contiguous()
        angle = torch.as_tensor(angle_deg, device=self.device).to(torch.float64).contiguous()
        assert env.shape == camera.shape == angle.shape
        out = torch.empty_like(angle)
        with torch.cuda.device(self.device):
            _check(self.lib, self.lib.mate_b200_fov_range(self.handle, _dptr(env), _dptr(camera), _dptr(angle), _dptr(out),
                                                          angle.numel(), self._stream()))
        return out

    def render(self, envs=None, size=800):
        """``rgb_array`` frames of the environments ``envs`` (``None`` = every environment, entry i = environment
        ``envs[i]``), drawn from the current state by a CUDA kernel (mate_b200_render, the picture is defined in
        ``include/mate_b200.h``): a new uint8 tensor ``[K, size, size, 3]`` on the simulator's device, written on the
        current stream without a synchronisation.  Host indices are checked here; the frame of an out-of-range device index
        is left unwritten."""
        size = check_render_size(size)
        index = self._index_map(envs, 'envs', None, 0, self.B)
        count = self.B if index is None else int(index.numel())
        out = torch.empty((count, size, size, 3), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _check(self.lib, self.lib.mate_b200_render(self.handle, _dptr(index), count, size, _dptr(out), self._stream()))
        return out

    def soft_coverage(self, auto_reset=True):
        """``AuxiliaryCameraRewards.compute_soft_coverage_scores`` for the current state and the camera-target masks
        of the last step: ``[B, Nc, Nt]`` float32 (mate_b200_soft_coverage).  With ``auto_reset`` the environments
        that were reset in the last step get zeros."""
        if self._aux is None:
            raise RuntimeError('soft_coverage needs a step / observe call with aux=True first')
        if getattr(self, '_soft', None) is None:
            self._soft = torch.zeros((self.B, self.nc, self.nt), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _check(self.lib, self.lib.mate_b200_soft_coverage(
                self.handle, _dptr(self._aux['mask_ct']), _dptr(self.done) if auto_reset else None, _dptr(self._soft), self._stream()))
        return self._soft

    def auxiliary_terms(self, soft_matrix=None):
        """Per-agent terms of the auxiliary-reward / training-information wrappers for the LAST step
        (mate_b200_auxiliary_terms): ``(cam_terms [B, Nc, CAM_TERMS], tgt_terms [B, Nt, TGT_TERMS])``; the
        ``soft_coverage_score`` columns are filled when ``soft_matrix`` (from :meth:`soft_coverage`) is given."""
        if self._aux is None:
            raise RuntimeError('auxiliary_terms needs a step / observe call with aux=True first')
        if getattr(self, '_terms', None) is None:
            self._terms = (torch.zeros((self.B, self.nc, _abi.CAM_TERMS), dtype=torch.float32, device=self.device),
                           torch.zeros((self.B, self.nt, _abi.TGT_TERMS), dtype=torch.float32, device=self.device))
        cam_terms, tgt_terms = self._terms
        with torch.cuda.device(self.device):
            _check(self.lib, self.lib.mate_b200_auxiliary_terms(
                self.handle, ctypes.byref(self._aux_struct), _dptr(self.rewards), _dptr(soft_matrix),
                _dptr(cam_terms) if self.nc else None, _dptr(tgt_terms), self._stream()))
        return cam_terms, tgt_terms

    def step_host(self, cam_act, tgt_act, out, auto_reset=True, rows_kept=False):
        """Host-buffer step: `cam_act`/`tgt_act` and the tensors in `out` (cam_obs, tgt_obs,
        rewards, done) are CPU tensors (pinned for full PCIe speed).  `rows_kept=True` promises that
        `out` is the tuple of the previous `step_host` call and has not been written to since
        (MATE_STEP_HOST_ROWS_KEPT, include/mate_b200.h): parts of the rows that stay zero are then not rewritten.
        cam_obs / tgt_obs have the simulator's ``observation_dtype``; the slot of a team that is not observed is ``None``."""
        cam_obs, tgt_obs, rewards, done = out
        for name, rows, observed in (('cam_obs', cam_obs if self.nc else None, self.cam_obs is not None),
                                     ('tgt_obs', tgt_obs, self.tgt_obs is not None)):
            if observed and rows is None and (name == 'tgt_obs' or self.nc):
                raise ValueError(f'step_host: {name} is None, but this simulator observes {self.observed_team!r}')
            if not observed and rows is not None:
                raise ValueError(f'step_host: {name} must be None, this simulator observes {self.observed_team!r} only')
            if rows is not None and rows.dtype != self.observation_dtype:   # the C call sees only a pointer
                raise ValueError(f'step_host: {name} is {rows.dtype}, the simulator writes {self.observation_dtype} rows')
        flags = (_abi.MATE_STEP_AUTO_RESET if auto_reset else 0) | (_abi.MATE_STEP_HOST_ROWS_KEPT if rows_kept else 0)
        _check(self.lib, self.lib.mate_b200_step_host(
            self.handle, _dptr(cam_act) if self.nc else None, _dptr(tgt_act),
            _dptr(cam_obs) if self.nc else None, _dptr(tgt_obs), _dptr(rewards), _dptr(done), flags))
        return out

    def get_state(self):
        arrays = _abi.alloc_state_arrays(self.B, self.nc, self.nt, self.no)
        view = _abi.state_view_from_arrays(arrays)
        _check(self.lib, self.lib.mate_b200_get_state(self.handle, ctypes.byref(view)))
        return arrays

    def set_state(self, arrays):
        arrays = dict(arrays)
        view = _abi.state_view_from_arrays(arrays)
        _check(self.lib, self.lib.mate_b200_set_state(self.handle, ctypes.byref(view)))

    def _index_map(self, index, name, length, low, high):
        """Environment / snapshot indices as an int32 tensor on the simulator's device (``None`` stays ``None``), checked
        by :func:`check_index_map`.  A device tensor is passed on without a synchronisation: the library's kernels skip
        entries that are out of range."""
        host = check_index_map(index, name, length, low, high)
        if index is None:
            return None
        if host is None:
            return index.to(self.device, torch.int32).contiguous()
        return torch.from_numpy(host.astype(np.int32)).to(self.device)

    def snapshot_bytes(self, count):
        """Bytes of the payload of a snapshot of ``count`` environments (mate_b200_snapshot_bytes)."""
        out = ctypes.c_uint64(0)
        _check(self.lib, self.lib.mate_b200_snapshot_bytes(self.handle, int(count), ctypes.byref(out)))
        return int(out.value)

    def save_state(self, envs=None):
        """Snapshot of the environments ``envs`` (``None`` = the whole batch, entry i = environment ``envs[i]``), saved on
        the device on the current stream (mate_b200_save_state): no synchronisation, no host copy of the state."""
        index = self._index_map(envs, 'envs', None, 0, self.B)
        with torch.cuda.device(self.device):
            count = self.B if index is None else int(index.numel())
            payload = torch.empty(self.snapshot_bytes(count), dtype=torch.uint8, device=self.device)
            info = _abi.MateSnapshotInfo()
            _check(self.lib, self.lib.mate_b200_save_state(self.handle, _dptr(index), count, _dptr(payload), ctypes.byref(info),
                                                           self._stream()))
        return StateSnapshot(payload, py_seed=self._seed, **{name: getattr(info, name) for name in _abi.SNAPSHOT_INFO_FIELDS})

    def load_state(self, snapshot, src=None, resume=False):
        """Load a snapshot on the current stream (mate_b200_load_state).  ``src=None``: environment d takes entry d (the
        snapshot holds the whole batch); otherwise environment d takes entry ``src[d]`` (``B`` indices) and a negative
        entry keeps environment d.  ``resume=True`` also takes the snapshot's seed and episode statistics, so the batch
        continues bit for bit where it was saved (whole-batch snapshots only)."""
        index = self._index_map(src, 'src', self.B, -(1 << 31), snapshot.count)
        with torch.cuda.device(self.device):
            payload = snapshot.payload
            if payload.device != self.device:
                payload = payload.to(self.device)
            payload = payload.contiguous()
            info = snapshot.info()
            _check(self.lib, self.lib.mate_b200_load_state(self.handle, _dptr(payload), ctypes.byref(info), _dptr(index),
                                                           _abi.MATE_LOAD_STATE_RESUME if resume else 0, self._stream()))
        if resume:
            self._seed = snapshot.py_seed

    def episode_stats(self, reset_after=False):
        with torch.cuda.device(self.device):
            _check(self.lib, self.lib.mate_b200_episode_stats(self.handle, _dptr(self._stats), int(reset_after),
                                                              self._stream()))
        return self._stats

    def host_leg_info(self):
        """(leg, row bytes on the link) of the last `step_host` call: 0 dense copy, 1 rows rebuilt from their non-zero
        chunks, 2 changes patched into kept rows (mate_b200_host_leg_info)."""
        leg, link = ctypes.c_int32(0), ctypes.c_uint64(0)
        _check(self.lib, self.lib.mate_b200_host_leg_info(self.handle, ctypes.byref(leg), ctypes.byref(link)))
        return int(leg.value), int(link.value)

    @property
    def launch_count(self):
        return int(self.lib.mate_b200_launch_count(self.handle))
