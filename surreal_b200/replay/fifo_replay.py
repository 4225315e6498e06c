"""FIFOReplay in HBM (drop-in for surreal/replay/fifo_replay.py:6-48).

Storage is a ring of ``memory_size + 3`` window records (SoA, record-major):
  obs  [C][n+1][D]  (row n is obs_next)   act [C][n][A]   pd [C][n][2A]   rew [C][n]   done [C][n]
with the queue control block {head, count, capacity, dropped, total_in, total_out} ALSO in device memory,
so on-device actors push windows without any host round trip.  Semantics are the reference's exactly:
arrival order out, silent drop of the OLDEST at capacity, ready when len >= batch_size.

``sample()`` pops the oldest ``batch_size`` windows and gathers them into the learner-facing batch
(the aggregator's layout, aggregator.py:176-183) as CUDA tensors."""
import ctypes as C

import numpy as np
import torch

from .. import _lib
from .._lib import check
from .base import Replay, gather_fields


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _st():
    from ..ops import _stream
    return _stream()


class FIFOReplay(Replay):
    def __init__(self, learner_config, env_config, session_config, index=0):
        super().__init__(learner_config, env_config, session_config, index)
        self.batch_size = self.learner_config.replay.batch_size
        self.memory_size = self.learner_config.replay.memory_size
        assert self.session_config.replay.max_puller_queue <= 10
        assert self.session_config.replay.max_prefetch_queue == 1
        assert not self.session_config.sender.flush_time
        assert self.session_config.sender.flush_iteration <= 10
        if not torch.cuda.is_available():
            raise RuntimeError('surreal_b200.FIFOReplay lives in HBM: a CUDA device is required')
        self.device = torch.device('cuda', torch.cuda.current_device())
        self.n_step = self.learner_config.algo.n_step
        from ..utils import record_obs_dim, obs_packed_dim, obs_is_pixel, obs_is_mixed, obs_layout
        self.D = record_obs_dim(self.learner_config, self.env_config)   # pixel frames: opaque 32-bit words; RNN: + LSTM cells
        self.obs_dim = obs_packed_dim(self.env_config.obs_spec)
        self.pixel_shape = tuple(self.env_config.obs_spec['pixel']['camera0']) if obs_is_pixel(self.env_config.obs_spec) else None
        # mixed observations: frame words + low-dim floats in one row (utils.obs_layout)
        self.layout = obs_layout(self.env_config.obs_spec) if obs_is_mixed(self.env_config.obs_spec) else None
        self.A = self.env_config.action_spec.dim[0]
        self.capacity = self.memory_size + 3                    # "+ 3 for a gentle buffering" (fifo_replay.py:27)
        C_, n, D, A = self.capacity, self.n_step, self.D, self.A
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=self.device)  # noqa: E731
        self.r_obs, self.r_act, self.r_pd = f(C_, n + 1, D), f(C_, n, A), f(C_, n, 2 * A)
        self.r_rew, self.r_done = f(C_, n), f(C_, n)
        L = _lib.lib()
        nb = int(L.sb200_fifo_state_bytes())                    # {head, count, capacity, dropped, int64 in, out, ...}
        assert nb >= 32 and nb % 4 == 0
        self.state = torch.zeros(nb // 4, dtype=torch.int32, device=self.device)
        self.state[2] = self.capacity
        self._idx = torch.zeros(max(self.batch_size, 1), dtype=torch.int32, device=self.device)
        self._status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._slots = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._pin = None
        self.check_underflow = True

    # -- control block ---------------------------------------------------------------------------------
    def _read_state(self):
        s = self.state.cpu().numpy()
        return dict(head=int(s[0]), count=int(s[1]), capacity=int(s[2]), dropped=int(s[3]),
                    total_in=int(s[4:6].view(np.int64)[0]), total_out=int(s[6:8].view(np.int64)[0]))

    def __len__(self):
        return self._read_state()['count']

    def start_sample_condition(self):
        return len(self) >= self.batch_size

    def evict(self):
        raise NotImplementedError('no support for eviction in FIFO mode')

    # -- host insert (external / CPU actors) -----------------------------------------------------------
    def insert(self, exp):
        """``exp``: the dict ExpSenderWrapperMultiStepMovingWindowWithInfo.send emits
        (exp_sender_wrapper.py:244-264): obs [n dicts], obs_next, actions, rewards, dones, persistent_infos."""
        n, D, A = self.n_step, self.D, self.A
        if self.layout is not None:
            from ..utils import pack_obs_rows
            flat = lambda o: pack_obs_rows(o, self.layout).reshape(-1)  # noqa: E731
        elif self.pixel_shape is not None:       # uint8 frame -> the same bytes viewed as float32 words
            flat = lambda o: np.ascontiguousarray(np.asarray(o['pixel']['camera0'], dtype=np.uint8)).reshape(-1).view(np.float32)  # noqa: E731
        else:
            flat = lambda o: np.concatenate([np.asarray(o['low_dim'][k], dtype=np.float32).reshape(-1)  # noqa: E731
                                             for k in o['low_dim']])
        assert len(exp['obs']) == n, 'window length %d != n_step %d' % (len(exp['obs']), n)
        rec = n * (D + A + 2 * A + 2) + D
        if self._pin is None:
            self._pin = torch.empty(rec, dtype=torch.float32, pin_memory=True)
            self._stage = torch.empty(rec, dtype=torch.float32, device=self.device)
        buf = self._pin.numpy()
        o = 0
        rows = np.zeros((n + 1, D), dtype=np.float32)
        od = self.obs_dim
        rows[:n, :od] = np.stack([flat(x) for x in exp['obs']])
        rows[n, :od] = flat(exp['obs_next'])
        if D > od and exp.get('onetime_infos'):                 # [h, c] of the window's first step (ppo_agent.py:133-137)
            Hh = (D - od) // 2
            rows[0, od:od + Hh] = np.asarray(exp['onetime_infos'][0], dtype=np.float32).reshape(-1)[:Hh]
            rows[0, od + Hh:] = np.asarray(exp['onetime_infos'][1], dtype=np.float32).reshape(-1)[:Hh]
        buf[o:o + (n + 1) * D] = rows.reshape(-1); o += (n + 1) * D
        buf[o:o + n * A] = np.stack(exp['actions']).astype(np.float32).reshape(-1); o += n * A
        buf[o:o + n * 2 * A] = np.stack([p[-1] for p in exp['persistent_infos']]).astype(np.float32).reshape(-1)
        o += n * 2 * A
        buf[o:o + n] = np.asarray(exp['rewards'], dtype=np.float32); o += n
        buf[o:o + n] = np.asarray(exp['dones'], dtype=np.float32)
        self._stage.copy_(self._pin, non_blocking=True)
        check(_lib.lib().sb200_fifo_push(_p(self.state), 1, _p(self._slots), _st()), 'sb200_fifo_push')
        slot = int(self._slots.item())
        s = self._stage
        o = 0
        self.r_obs[slot].view(-1).copy_(s[o:o + (n + 1) * D]); o += (n + 1) * D
        self.r_act[slot].view(-1).copy_(s[o:o + n * A]); o += n * A
        self.r_pd[slot].view(-1).copy_(s[o:o + n * 2 * A]); o += n * 2 * A
        self.r_rew[slot].copy_(s[o:o + n]); o += n
        self.r_done[slot].copy_(s[o:o + n])

    # -- sample ------------------------------------------------------------------------------------------
    def sample(self, batch_size, out=None):
        """Pop the ``batch_size`` oldest windows (arrival order) -> aggregated device batch."""
        assert batch_size <= self.memory_size
        L = _lib.lib()
        n, D, A = self.n_step, self.D, self.A
        if self._idx.numel() < batch_size:
            self._idx = torch.zeros(batch_size, dtype=torch.int32, device=self.device)
        check(L.sb200_fifo_pop(_p(self.state), batch_size, _p(self._idx), _p(self._status), _st()), 'sb200_fifo_pop')
        if out is None:
            f = lambda *s: torch.empty(*s, dtype=torch.float32, device=self.device)  # noqa: E731
            out = dict(obs_full=f(batch_size, n + 1, D), actions=f(batch_size, n, A), pd=f(batch_size, n, 2 * A),
                       rewards=f(batch_size, n), dones=f(batch_size, n))
        gather_fields([(self.r_obs, out['obs_full'], (n + 1) * D), (self.r_act, out['actions'], n * A),
                       (self.r_pd, out['pd'], n * 2 * A), (self.r_rew, out['rewards'], n), (self.r_done, out['dones'], n)],
                      self._idx, None, batch_size)                      # all five fields: one launch
        if self.check_underflow and int(self._status.item()) != 0:      # host sync; the engine polls
            raise IndexError('pop from a FIFO replay holding fewer than %d windows' % batch_size)   # len() instead
        obs_full = out['obs_full']
        if self.layout is not None:
            # views into the batch: uint8 frames [B, n(+1), C, H, W] and one [B, n(+1), width] view per low-dim key
            from ..utils import mixed_obs_views
            return {'obs': mixed_obs_views(obs_full[:, :n], self.layout), 'obs_next': mixed_obs_views(obs_full[:, n:], self.layout),
                    'obs_full': obs_full, 'actions': out['actions'], 'rewards': out['rewards'], 'dones': out['dones'],
                    'persistent_infos': [out['pd']], 'onetime_infos': None}
        if self.pixel_shape is not None:
            fr = obs_full.view(torch.uint8).view(batch_size, n + 1, *self.pixel_shape)
            return {'obs': {'pixel': {'camera0': fr[:, :n]}}, 'obs_next': {'pixel': {'camera0': fr[:, n:]}},
                    'obs_full': obs_full, 'actions': out['actions'], 'rewards': out['rewards'], 'dones': out['dones'],
                    'persistent_infos': [out['pd']], 'onetime_infos': None}
        od = self.obs_dim
        onetime = None
        if D > od:                 # RNN policy: the LSTM cells of the window's first step ride behind the observation
            Hh = (D - od) // 2
            onetime = [obs_full[:, 0, od:od + Hh].unsqueeze(1), obs_full[:, 0, od + Hh:od + 2 * Hh].unsqueeze(1)]
        return {'obs': {'low_dim': {'flat_inputs': obs_full[:, :n, :od]}},
                'obs_next': {'low_dim': {'flat_inputs': obs_full[:, n:, :od]}},
                'obs_full': obs_full, 'actions': out['actions'], 'rewards': out['rewards'], 'dones': out['dones'],
                'persistent_infos': [out['pd']], 'onetime_infos': onetime}
