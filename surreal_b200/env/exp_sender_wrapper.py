"""Experience-sender wrappers for BATCHED device-resident envs (mirror of
surreal/env/exp_sender_wrapper.py:72-112,153-264).

The reference keeps one Python deque per actor process and ships finished windows / n-step transitions
through pyarrow + ZeroMQ to the replay server.  Here the N deques are HBM arrays, the "send" is a kernel
that copies the record into the HBM replay's ring in (step, actor) order, and the md5 de-duplication of
overlapping windows (exp_sender.py:10-59) has nothing left to do."""
import ctypes as C

import torch

from .. import _lib
from .._lib import check
from ..distributed import LocalHub
from ..session import ConfigError
from ..utils import obs_flat, obs_is_mixed, obs_packed_dim


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _st():
    from ..ops import _stream
    return _stream()


class _WrapperBase:
    def __init__(self, env, learner_config, session_config, replay=None, obs_extra=0):
        self.env = env
        self.learner_config = learner_config
        self.session_config = session_config
        self.replay = replay if replay is not None else LocalHub.get(session_config).replays.get(0)
        if self.replay is None:
            raise RuntimeError('no replay registered for this session: construct the Replay before the agent '
                               'wraps its env (the ZeroMQ collector address of the reference is gone)')
        # mixed observations (frame + low-dim): the rows are packed in the layout of utils.obs_layout, in this spec's key order
        spec = env.observation_spec() if hasattr(env, 'observation_spec') else None
        self.obs_spec = spec if (spec is not None and obs_is_mixed(spec)) else None
        D = obs_packed_dim(self.obs_spec) if self.obs_spec is not None else env.D
        self.N, self.D, self.A = env.N, D + int(obs_extra), env.A
        # extra trailing floats per observation row, filled by ``obs_augment(rows [N, env.D]) -> [N, D]`` (an RNN agent appends
        # its LSTM cells; utils.record_obs_dim)
        self.obs_extra, self.obs_augment = int(obs_extra), None
        # a batched HOST env (numpy in / numpy out, attributes N, D, A) has no device: the staging lives with the replay
        self.device = env.device if hasattr(env, 'device') else self.replay.device
        self.host_env = not hasattr(env, 'device')
        self._pins, self._devs = {}, {}
        self._last_obs_host, self._last_obs_dev = None, None
        if not hasattr(env, 'step_counter'):
            self.step_counter = torch.zeros(1, dtype=torch.int64, device=self.device)   # Philox step counter

    def _h2d(self, name, arr, shape):
        """numpy -> device through a persistent pinned staging buffer (skipped when ``arr`` already is pinned)."""
        import numpy as np
        dev = self._devs.get(name)
        if dev is None:
            dev = self._devs[name] = torch.zeros(*shape, dtype=torch.float32, device=self.device)
        src = None
        if isinstance(arr, np.ndarray) and arr.dtype == np.float32 and arr.flags['C_CONTIGUOUS'] and arr.flags['WRITEABLE']:
            t = torch.from_numpy(arr)
            if t.is_pinned():
                src = t.view(*shape)
        if src is None:
            pin = self._pins.get(name)
            if pin is None:
                pin = self._pins[name] = torch.empty(*shape, dtype=torch.float32, pin_memory=True)
            pin.numpy()[...] = np.asarray(arr, dtype=np.float32).reshape(shape)
            src = pin
        dev.copy_(src, non_blocking=True)
        return dev

    def _dev(self, name, shape):
        dev = self._devs.get(name)
        if dev is None:
            dev = self._devs[name] = torch.zeros(*shape, dtype=torch.float32, device=self.device)
        return dev

    def _pinned(self, name, arr, shape):
        """Address (c_void_p) of ``arr`` if it already lives in pinned memory, else of a pinned staging copy."""
        import numpy as np
        if isinstance(arr, np.ndarray) and arr.dtype == np.float32 and arr.flags['C_CONTIGUOUS'] and arr.flags['WRITEABLE'] \
                and torch.from_numpy(arr).is_pinned():
            return C.c_void_p(arr.ctypes.data)
        pin = self._pins.get(name)
        if pin is None:
            pin = self._pins[name] = torch.empty(*shape, dtype=torch.float32, pin_memory=True)
        pin.numpy()[...] = np.asarray(arr, dtype=np.float32).reshape(shape)
        return C.c_void_p(pin.data_ptr())

    def _aug(self, o):
        return self.obs_augment(o, 0) if (self.obs_extra and self.obs_augment is not None) else o

    def _aug_next(self, o):
        return self.obs_augment(o, 1) if (self.obs_extra and self.obs_augment is not None) else o

    def cached_device_obs(self, obs_arr):
        """The device copy of the observation the last step() returned (the agent's next act() input), if
        ``obs_arr`` is that very array: saves the second H2D of the same 256 KB."""
        return self._last_obs_dev if (obs_arr is not None and obs_arr is self._last_obs_host) else None

    @property
    def unwrapped(self):
        return getattr(self.env, 'unwrapped', self.env)

    def __getattr__(self, k):
        return getattr(self.env, k)


class ExpSenderWrapperMultiStepMovingWindowWithInfo(_WrapperBase):
    """n_step windows with stride (exp_sender_wrapper.py:153-264) -> FIFOReplay ring."""

    def __init__(self, env, learner_config, session_config, replay=None, obs_extra=0):
        super().__init__(env, learner_config, session_config, replay, obs_extra=obs_extra)
        self.n_step = self.learner_config.algo.n_step
        self.stride = self.learner_config.algo.stride
        if self.stride < 1:
            raise ConfigError('stride {} for experience generation cannot be less than 1'.format(self.stride))
        N, n, D, A = self.N, self.n_step, self.D, self.A
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=self.device)  # noqa: E731
        self.stage_pos = torch.zeros(N, dtype=torch.int32, device=self.device)
        self.stage_obs, self.stage_act, self.stage_pd = f(N, n + 1, D), f(N, n, A), f(N, n, 2 * A)
        self.stage_rew, self.stage_done = f(N, n), f(N, n)
        self._dest = torch.zeros(N, dtype=torch.int32, device=self.device)
        self._slots_ready = False      # the agent's sampling kernel already assigned this step's replay slots
        self.fuse_launches = True      # sample+assign / env+commit: 3 launches per step instead of 5 (same results)
        self.persistent_rollout = True  # device env + supported policy: whole chunks in ONE launch (agent.rollout_chunk)
        self._outbox = {}
        r = self.replay
        assert (r.n_step, r.D, r.A) == (n, D, A), 'replay record shape does not match the env / n_step'

    def reset(self):
        obs, info = self.env.reset()
        self.stage_pos.zero_()                                     # deque.clear() (exp_sender_wrapper.py:204-207)
        o = obs_flat(obs, self.obs_spec)
        if self.host_env:
            d = self._h2d('obs', o, (self.N, self.D))
            self.stage_obs[:, 0].copy_(d)
            self._last_obs_host, self._last_obs_dev = o, d
        else:
            self.stage_obs[:, 0].copy_(self._aug(o))
        return obs, info

    def rollout_outbox(self, T):
        """Buffers of the persistent rollout kernel for chunks of T steps: per-actor outbox of finished windows (in
        the replay's record layout), their completion steps, and the commit pass's scratch.  None when the outbox
        would not be worth its memory (tiny strides)."""
        key = int(T)
        if key in self._outbox:
            return self._outbox[key]
        N, n, D, A = self.N, self.n_step, self.D, self.A
        W = T // self.stride + 2
        rec_bytes = 4 * ((n + 1) * D + n * A + n * 2 * A + 2 * n)
        ob = None
        if N * W * rec_bytes <= 4 << 30:
            f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=self.device)  # noqa: E731
            z = lambda k: torch.zeros(k, dtype=torch.int32, device=self.device)      # noqa: E731
            ob = dict(W=W, o_obs=f(N * W, n + 1, D), o_act=f(N * W, n, A), o_pd=f(N * W, n, 2 * A), o_rew=f(N * W, n),
                      o_done=f(N * W, n), ev_step=z(N * W), ev_count=z(N),
                      scratch=z(int(_lib.lib().sb200_ppo_rollout_scratch_ints(N, W, T))))
        self._outbox[key] = ob
        return ob

    def slot_assignment_args(self):
        """For PPOAgent.act: (fifo_state, dest) of sb200_ppo_sample_assign_f32, which folds this step's slot
        assignment into the sampling launch.  The following step() then skips its own assignment pass."""
        self._slots_ready = True
        return self.replay.state, self._dest

    def step(self, action):
        """``action`` = (action_choice, action_info) as PPOAgent.act returns in training mode; the agent has
        already staged action / pd rows for this step (sb200_ppo_sample[_assign]_f32)."""
        a = action[0] if isinstance(action, tuple) else action
        r = self.replay
        ready, self._slots_ready = self._slots_ready, False
        if ready and hasattr(self.env, 'step_and_commit_window') and not self.obs_extra:
            return self.env.step_and_commit_window(a, self)        # env step + commit in ONE launch
        obs, reward, done, info = self.env.step(a)
        o = obs_flat(obs, self.obs_spec)
        on = obs_flat(info['obs_next'], self.obs_spec) if (isinstance(info, dict) and 'obs_next' in info) else o
        if self.host_env and self.obs_extra:
            raise NotImplementedError('RNN policy with a host env: stage the windows with replay.insert (onetime_infos) instead')
        if self.host_env:
            # host env: this step's successor observation / reward / done cross PCIe here (256 KB + 8 KB), issued with
            # the staging kernels from ONE C call; the device copy of the next observation is handed to the agent's
            # next act() (cached_device_obs)
            h_o, h_on = self._pinned('obs', o, (self.N, self.D)), None
            h_on = h_o if on is o else self._pinned('obs_next', on, (self.N, self.D))
            h_r, h_d = self._pinned('rew', reward, (self.N,)), self._pinned('done', done, (self.N,))
            d_o, d_on = self._dev('obs', (self.N, self.D)), self._dev('obs_next', (self.N, self.D))
            d_r, d_d = self._dev('rew', (self.N,)), self._dev('done', (self.N,))
            check(_lib.lib().sb200_ppo_window_step_host_f32(
                h_on, h_o, h_r, h_d, _p(d_on), _p(d_o), _p(d_r), _p(d_d), self.N, self.n_step, self.stride, self.D,
                self.A, _p(self.stage_pos), _p(self.stage_obs), _p(self.stage_act), _p(self.stage_pd),
                _p(self.stage_rew), _p(self.stage_done), _p(self._dest), _p(r.state), _p(r.r_obs), _p(r.r_act),
                _p(r.r_pd), _p(r.r_rew), _p(r.r_done), _p(self.step_counter), int(ready), _st()),
                'sb200_ppo_window_step_host_f32')
            self._last_obs_host, self._last_obs_dev = o, d_o
            return obs, reward, done, info
        if self.obs_extra:
            # both rows get the cells the agent holds NOW, i.e. before it acts on the next observation; `on` and `o` differ
            # only where an episode ended
            same = on is o
            o = self._aug(o)
            on = o if same else self._aug_next(on)
        check(_lib.lib().sb200_ppo_window_step_f32(
            _p(on), _p(o), _p(reward), _p(done), self.N, self.n_step,
            self.stride, self.D, self.A, _p(self.stage_pos), _p(self.stage_obs), _p(self.stage_act),
            _p(self.stage_pd), _p(self.stage_rew), _p(self.stage_done), _p(self._dest), _p(r.state), _p(r.r_obs),
            _p(r.r_act), _p(r.r_pd), _p(r.r_rew), _p(r.r_done), _p(self.step_counter), int(ready), _st()),
            'sb200_ppo_window_step_f32')
        return obs, reward, done, info


class ExpSenderWrapperSSARNStepBootstrap(_WrapperBase):
    """n-step bootstrapped SSAR transitions (exp_sender_wrapper.py:72-112) -> UniformReplay ring."""

    def __init__(self, env, learner_config, session_config, replay=None):
        super().__init__(env, learner_config, session_config, replay)
        self.n_step = self.learner_config.algo.n_step
        self.gamma = self.learner_config.algo.gamma
        N, n, D, A = self.N, self.n_step, self.D, self.A
        self.dq_len = torch.zeros(N, dtype=torch.int32, device=self.device)
        self.dq_obs = torch.zeros(N, n, D, device=self.device)
        self.dq_act = torch.zeros(N, n, A, device=self.device)
        self.dq_rew = torch.zeros(N, n, dtype=torch.float64, device=self.device)
        self._dest = torch.zeros(N, dtype=torch.int32, device=self.device)
        self._emit = torch.zeros(N, device=self.device)
        self._obs = torch.zeros(N, D, device=self.device)

    def reset(self):
        obs, info = self.env.reset()
        self.dq_len.zero_()
        self._obs.copy_(obs['low_dim']['flat_inputs'])
        return obs, info

    def step(self, action):
        obs, reward, done, info = self.env.step(action)
        r = self.replay
        check(_lib.lib().sb200_ssar_step_f32(
            _p(self._obs), _p(action), _p(info['obs_next']), _p(reward), _p(done), self.N, self.n_step,
            float(self.gamma), self.D, self.A, _p(self.dq_len), _p(self.dq_obs), _p(self.dq_act), _p(self.dq_rew),
            _p(self._dest), _p(self._emit), _p(r.state), _p(r.r_obs), _p(r.r_obs_next), _p(r.r_act), _p(r.r_rew),
            _p(r.r_done), _p(self.env.step_counter), _st()), 'sb200_ssar_step_f32')
        r.mark_device_inserts()
        self._obs.copy_(obs['low_dim']['flat_inputs'])             # s_t of the next transition (reset obs where done)
        return obs, reward, done, info
