"""Small host-side helpers shared by the plugin classes (constructor protocol, timers, trackers).

AutoInitializeMeta mirrors the reference's constructor protocol (surreal/utils/common.py:232-275):
``_initialize()`` runs after the most-derived ``__init__``.  The timers keep the names the reference
reports under (learner/base.py:160-162, replay/base.py:139-141)."""
import logging
import threading
import time
from contextlib import contextmanager


class AutoInitializeMeta(type):
    def __call__(cls, *args, **kwargs):
        obj = super().__call__(*args, **kwargs)
        if not hasattr(obj, '_initialize'):
            raise AssertionError('AutoInitializeMeta requires that subclass implements _initialize()')
        obj._initialize()
        return obj


class MovingAverageRecorder:
    """Exponential moving average with bias correction (first value seeds the average)."""

    def __init__(self, decay=0.95):
        self.decay = decay
        self.cum_value = 0.0
        self.normalization = 0.0
        self._lock = threading.Lock()

    def add_value(self, value):
        with self._lock:
            self.cum_value = self.cum_value * self.decay + value
            self.normalization = self.normalization * self.decay + 1.0
            return self.cum_value / self.normalization

    def cur_value(self):
        with self._lock:
            return self.cum_value / self.normalization if self.normalization > 0 else 0.0


class TimeRecorder:
    def __init__(self, decay=0.9995, max_seconds=10):
        self.moving_average = MovingAverageRecorder(decay)
        self.max_seconds = max_seconds
        self.started = False

    @contextmanager
    def time(self):
        t0 = time.time()
        yield None
        self.moving_average.add_value(min(self.max_seconds, time.time() - t0))

    def start(self):
        if self.started:
            raise RuntimeError('Starting a started timer')
        self.pre_time = time.time()
        self.started = True

    def lap(self):
        if not self.started:
            raise RuntimeError('Stopping a timer that is not started')
        now = time.time()
        self.moving_average.add_value(min(self.max_seconds, now - self.pre_time))
        self.pre_time = now

    def stop(self):
        self.lap()
        self.started = False

    @property
    def avg(self):
        return self.moving_average.cur_value()


class PeriodicTracker:
    """True once every ``period`` increments (surreal/session/tracker.py:10-44)."""

    def __init__(self, period, init_value=0, init_endpoint=0):
        assert isinstance(period, int) and period > 0
        self.period, self.value, self._endpoint = period, init_value, init_endpoint

    def _update(self):
        if self.value >= self._endpoint + self.period:
            self._endpoint += (self.value - self._endpoint) // self.period * self.period
            return True
        return False

    def track_increment(self, incr=1):
        self.value += incr
        return self._update()

    def track_absolute(self, value):
        self.value = value
        return self._update()


class TimedTracker:
    """True when at least ``interval`` seconds passed since the last True (utils/common.py:590-610)."""

    def __init__(self, interval):
        self.interval = interval
        self.last_time = time.time()

    def track_increment(self):
        now = time.time()
        if now - self.last_time >= self.interval:
            self.last_time = now
            return True
        return False


class ScalarSink:
    """Stand-in for the tensorplex client: keeps the last scalars per step (``add_scalars`` is the only
    call the hot path makes, learner/base.py:611; the ZMQ->TensorBoard multiplexer is out of scope)."""

    def __init__(self, name='learner'):
        self.name = name
        self.last = {}
        self.history = []
        self.keep_history = False

    def add_scalars(self, tag_to_scalar, global_step=None):
        self.last = dict(tag_to_scalar)
        if self.keep_history:
            self.history.append((global_step, dict(tag_to_scalar)))


def get_logger(name):
    log = logging.getLogger('surreal_b200.' + name)
    if not log.handlers:
        h = logging.StreamHandler()
        h.setFormatter(logging.Formatter('[%(name)s] %(message)s'))
        log.addHandler(h)
        log.setLevel(logging.WARNING)
    return log


def obs_is_pixel(obs_spec):
    """True for a spec with a camera frame ({'pixel': {'camera0': (C, H, W)}}, docs/env.md:79-108), with or without
    low-dim inputs next to it (see obs_is_mixed)."""
    return 'pixel' in obs_spec and len(obs_spec['pixel']) > 0


def obs_is_mixed(obs_spec):
    """True for a camera frame together with low-dim inputs (the robosuite observation, ppo_configs.py:111-114)."""
    return obs_is_pixel(obs_spec) and 'low_dim' in obs_spec and len(obs_spec['low_dim']) > 0


def obs_layout(obs_spec):
    """Where each part of one observation sits in a record row (see obs_packed_dim), in 32-bit words:

        width        words per row
        frame_shape  (C, H, W) of the camera frame, or None
        frame_bytes  C*H*W (0 without a frame); the frame starts at word 0
        low_dim_off  first word of the low-dim floats
        low_dim      number of low-dim floats
        keys         [(key, word offset, width)] of the low-dim inputs, in obs_spec order"""
    frame_shape, frame_bytes = None, 0
    if obs_is_pixel(obs_spec):
        frame_shape = tuple(int(v) for v in obs_spec['pixel']['camera0'])
        frame_bytes = 1
        for v in frame_shape:
            frame_bytes *= v
        if frame_bytes % 16 != 0:
            raise ValueError('pixel observations need C*H*W to be a multiple of 16 bytes, got %s' % (frame_shape,))
    off = frame_bytes // 4
    keys = []
    for k, v in (obs_spec['low_dim'].items() if 'low_dim' in obs_spec else ()):
        keys.append((k, off, int(v[0])))
        off += int(v[0])
    low_dim = off - frame_bytes // 4
    width = (off + 3) // 4 * 4 if (frame_bytes and low_dim) else off
    return dict(width=width, frame_shape=frame_shape, frame_bytes=frame_bytes, low_dim_off=frame_bytes // 4, low_dim=low_dim,
                keys=keys)


def obs_packed_dim(obs_spec):
    """Floats per observation in the HBM staging / replay records.

    Low-dim observations: the concatenated feature width.  Pixel observations: the uint8 frame is carried as an opaque run of
    C*H*W/4 32-bit words (only ever COPIED by the windowing / replay kernels, never computed on), so frames stay uint8 in HBM:
    28 224 B per 4x84x84 frame.  Mixed observations (a frame and low-dim inputs): the frame words first, at word 0, then the
    low-dim floats concatenated in obs_spec['low_dim'] order, then zero padding up to a multiple of 4 words (at most 12
    bytes).  Frames are a multiple of 16 bytes, so both parts and every row start 16-byte aligned for the vector loads of
    the replay, stem and MLP kernels.  obs_layout gives the offsets; nothing else computes them."""
    return obs_layout(obs_spec)['width']


def pack_obs_rows(obs, layout, out=None):
    """Host observation dict (numpy, leading dims [...]) -> float32 record rows [..., width] in the layout of obs_layout.
    Mixed / pixel frames are copied as raw bytes; ``out`` (e.g. a pinned buffer's numpy view) receives the rows."""
    import numpy as np
    lead = None
    if layout['frame_bytes']:
        fr = np.ascontiguousarray(np.asarray(obs['pixel']['camera0'], dtype=np.uint8))
        lead = fr.shape[:fr.ndim - len(layout['frame_shape'])]
    else:
        k0 = layout['keys'][0][0]
        a = np.asarray(obs['low_dim'][k0])
        lead = a.shape[:-1]
    if out is None:
        out = np.zeros(lead + (layout['width'],), dtype=np.float32)
    rows = out.reshape(-1, layout['width'])
    if layout['frame_bytes']:
        rows[:, :layout['frame_bytes'] // 4] = fr.reshape(-1, layout['frame_bytes']).view(np.float32)
    for k, off, w in layout['keys']:
        rows[:, off:off + w] = np.asarray(obs['low_dim'][k], dtype=np.float32).reshape(-1, w)
    return out


def mixed_obs_views(rows, layout):
    """Record rows [..., width] (float32 tensor, contiguous last dim) -> the observation dict of a mixed spec as VIEWS into
    them: {'pixel': {'camera0': uint8 [..., C, H, W]}, 'low_dim': {key: [..., width_k]}}."""
    import torch
    u8 = rows.view(torch.uint8)[..., :layout['frame_bytes']]
    fr = u8.unflatten(-1, layout['frame_shape'])
    return {'pixel': {'camera0': fr}, 'low_dim': {k: rows[..., off:off + w] for k, off, w in layout['keys']}}


def obs_flat(obs, obs_spec=None):
    """The per-actor rows [N, packed_dim] the staging kernels copy: the low-dim feature tensor, or the uint8 frames viewed
    as 32-bit words.  A mixed observation dict (frame + low-dim) is already packed when it comes from a device env
    (SyntheticMixedEnv hands out views into its record rows; those rows are returned); a host (numpy) one is packed into
    a new array in the layout of obs_layout (``obs_spec`` gives the key order, else the dict's own order)."""
    import torch
    if isinstance(obs, dict):
        mixed = 'pixel' in obs and len(obs['pixel']) > 0 and 'low_dim' in obs and len(obs['low_dim']) > 0
        if mixed:
            fr = obs['pixel']['camera0']
            if obs_spec is None:
                obs_spec = {'pixel': {'camera0': tuple(fr.shape[-3:])},
                            'low_dim': {k: (v.shape[-1],) for k, v in obs['low_dim'].items()}}
            lay = obs_layout(obs_spec)
            if not isinstance(fr, torch.Tensor):
                return pack_obs_rows(obs, lay)
            return _packed_rows_of(fr, obs, lay)
        if 'low_dim' in obs and len(obs['low_dim']) > 0:
            return obs['low_dim']['flat_inputs'] if 'flat_inputs' in obs['low_dim'] else next(iter(obs['low_dim'].values()))
        fr = obs['pixel']['camera0']
        return fr.reshape(fr.shape[0], -1).view(torch.float32)
    return obs


def _packed_rows_of(fr, obs, lay):
    """The record rows [N, width] a device mixed observation dict views into (frame at word 0 of each row)."""
    import torch
    N, W = fr.shape[0], lay['width']
    ok = fr.dtype == torch.uint8 and fr.is_cuda and fr.stride(0) == 4 * W and fr.storage_offset() % 4 == 0
    if ok:
        rows = torch.empty(0, dtype=torch.float32, device=fr.device)
        rows.set_(fr.untyped_storage(), fr.storage_offset() // 4, (N, W), (W, 1))
        for k, off, w in lay['keys']:
            v = obs['low_dim'][k]
            ok = ok and isinstance(v, torch.Tensor) and v.data_ptr() == rows.data_ptr() + 4 * off and v.stride(0) == W
    if not ok:
        raise ValueError('a device mixed observation must be views into packed record rows (SyntheticMixedEnv); pass host '
                         'arrays to have them packed')
    return rows


def record_obs_dim(learner_config, env_config):
    """Floats per observation row of the HBM staging / replay records and the learner's batch buffers: obs_packed_dim, plus
    -- for an RNN policy -- 2 * rnn_hidden trailing floats that carry the actor's LSTM cells (h | c) BEFORE it acted on that
    observation.  The reference ships the cells of a window's first step as ``onetime_infos``
    (ppo_agent.py:133-137, exp_sender_wrapper.py:244-264); here they simply ride with every observation row."""
    d = obs_packed_dim(env_config.obs_spec)
    rnn = learner_config.algo.rnn if 'rnn' in learner_config.algo else None
    if rnn is not None and rnn.if_rnn_policy:
        d += 2 * int(rnn.rnn_hidden)
    return d
