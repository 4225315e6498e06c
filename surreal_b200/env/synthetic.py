"""Batched, device-resident synthetic environment of the benchmark configs (SURVEY.md §8d, cfg 2/3/5):

    s' = tanh(Ws s + Wa a) + 0.01 xi,   r = -|s|^2 / D + 0.1 xi',   Ws, Wa ~ N(0, 1/sqrt(D)),  s0 ~ N(0,1)

with the episode cap of MaxStepWrapper (surreal/env/wrapper.py:142-163) folded in: ``done`` when an
actor's episode reaches ``limit_episode_length``; done actors auto-reset.  All N actors advance with ONE
kernel launch and every tensor stays in HBM.  The gym / MuJoCo / robosuite adapters of surreal/env are out
of scope (SURVEY §2 row 6); an external CPU env can still drive ``agent.act`` with numpy observations."""
import ctypes as C

import torch

from .. import _lib
from .._lib import check
from ..ops import _stream


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class SyntheticEnv:
    metadata = {}
    graph_safe = True          # obs IS the state buffer: fixed address, no host logic inside step()

    def __init__(self, num_envs, obs_dim=64, action_dim=8, limit_episode_length=200, seed=0, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError('SyntheticEnv is device-resident: a CUDA device is required')
        self.device = torch.device(device if device is not None else ('cuda:%d' % torch.cuda.current_device()))
        self.N, self.D, self.A = num_envs, obs_dim, action_dim
        self.max_steps = int(limit_episode_length)
        self.seed = int(seed)
        g = torch.Generator().manual_seed(self.seed)
        scale = 1.0 / (obs_dim ** 0.5)
        self.Ws = (torch.randn(obs_dim, obs_dim, generator=g) * scale).to(self.device)
        self.Wa = (torch.randn(obs_dim, action_dim, generator=g) * scale).to(self.device)
        self.WsT, self.WaT = self.Ws.t().contiguous(), self.Wa.t().contiguous()     # kernel layout (k-major)
        self._g = torch.Generator().manual_seed(self.seed + 1)
        self.state = torch.zeros(num_envs, obs_dim, device=self.device)
        self.ep_step = torch.zeros(num_envs, dtype=torch.int32, device=self.device)
        self.obs_next = torch.zeros(num_envs, obs_dim, device=self.device)
        self.reward = torch.zeros(num_envs, device=self.device)
        self.done = torch.zeros(num_envs, device=self.device)
        self.step_counter = torch.zeros(1, dtype=torch.int64, device=self.device)   # shared Philox counter
        self._own_counter = True

    def observation_spec(self):
        return {'low_dim': {'flat_inputs': (self.D,)}}

    def action_spec(self):
        return {'dim': (self.A,), 'type': 'continuous'}

    def reset(self):
        self.state.copy_(torch.randn(self.N, self.D, generator=self._g).to(self.device))
        self.ep_step.zero_()
        return {'low_dim': {'flat_inputs': self.state}}, {}

    def step(self, action):
        """action: [N, A] CUDA tensor.  Returns (obs, reward, done, info): obs is what every actor observes NEXT
        (already reset where done); ``info['obs_next']`` is the true successor (terminal where done)."""
        if isinstance(action, tuple):
            action = action[0]
        check(_lib.lib().sb200_synth_env_step_f32(
            _p(self.state), _p(action), _p(self.WsT), _p(self.WaT), self.N, self.D, self.A, self.max_steps,
            _p(self.ep_step), self.seed + 7, _p(self.step_counter), _p(self.obs_next), _p(self.reward), _p(self.done),
            _stream()), 'sb200_synth_env_step_f32')
        return {'low_dim': {'flat_inputs': self.state}}, self.reward, self.done, {'obs_next': self.obs_next}

    def step_and_commit_window(self, action, w):
        """step() fused with the commit half of ExpSenderWrapperMultiStepMovingWindowWithInfo.step (``w``), for
        steps whose replay slots the sampling kernel has already assigned."""
        r = w.replay
        check(_lib.lib().sb200_synth_env_window_step_f32(
            _p(self.state), _p(action), _p(self.WsT), _p(self.WaT), self.N, self.D, self.A, self.max_steps,
            _p(self.ep_step), self.seed + 7, _p(self.step_counter), _p(self.obs_next), _p(self.reward), _p(self.done),
            w.n_step, w.stride, _p(w.stage_pos), _p(w.stage_obs), _p(w.stage_act), _p(w.stage_pd), _p(w.stage_rew),
            _p(w.stage_done), _p(w._dest), _p(r.r_obs), _p(r.r_act), _p(r.r_pd), _p(r.r_rew), _p(r.r_done),
            _stream()), 'sb200_synth_env_window_step_f32')
        return {'low_dim': {'flat_inputs': self.state}}, self.reward, self.done, {'obs_next': self.obs_next}

    def close(self):
        pass


class SyntheticPixelEnv:
    """Batched device-resident PIXEL env of BASELINE configs[3] (SURVEY §8d cfg 4): every step each actor observes a fresh
    uint8 frame [C, H, W] of uniform random bytes; reward = -mean(a^2) + 0.1 xi; episodes end at ``limit_episode_length``.
    The staging / replay kernels see a frame as C*H*W/4 opaque 32-bit words (``D``), so frames stay uint8 in HBM."""
    metadata = {}
    graph_safe = True

    def __init__(self, num_envs, frame_shape=(4, 84, 84), action_dim=8, limit_episode_length=200, seed=0, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError('SyntheticPixelEnv is device-resident: a CUDA device is required')
        self.device = torch.device(device if device is not None else ('cuda:%d' % torch.cuda.current_device()))
        self.N, self.A = num_envs, action_dim
        self.frame_shape = tuple(int(v) for v in frame_shape)
        self.frame_bytes = 1
        for v in self.frame_shape:
            self.frame_bytes *= v
        assert self.frame_bytes % 16 == 0, 'C*H*W must be a multiple of 16 bytes'
        self.D = self.frame_bytes // 4
        self.max_steps = int(limit_episode_length)
        self.seed = int(seed)
        self._g = torch.Generator().manual_seed(self.seed + 1)
        self.state = torch.zeros(num_envs, self.frame_bytes, dtype=torch.uint8, device=self.device)
        self.obs_next = torch.zeros_like(self.state)
        self.ep_step = torch.zeros(num_envs, dtype=torch.int32, device=self.device)
        self.reward = torch.zeros(num_envs, device=self.device)
        self.done = torch.zeros(num_envs, device=self.device)
        self.step_counter = torch.zeros(1, dtype=torch.int64, device=self.device)

    def _obs(self, frames):
        return {'pixel': {'camera0': frames.view(self.N, *self.frame_shape)}}

    def observation_spec(self):
        return {'pixel': {'camera0': self.frame_shape}}

    def action_spec(self):
        return {'dim': (self.A,), 'type': 'continuous'}

    def reset(self):
        self.state.copy_(torch.randint(0, 256, (self.N, self.frame_bytes), generator=self._g, dtype=torch.uint8).to(self.device))
        self.ep_step.zero_()
        return self._obs(self.state), {}

    def step(self, action):
        if isinstance(action, tuple):
            action = action[0]
        check(_lib.lib().sb200_synth_pixel_env_step_u8(
            _p(self.state), _p(action), self.N, self.frame_bytes, self.A, self.max_steps, _p(self.ep_step), self.seed + 7,
            _p(self.step_counter), _p(self.obs_next), _p(self.reward), _p(self.done), _stream()), 'sb200_synth_pixel_env_step_u8')
        return self._obs(self.state), self.reward, self.done, {'obs_next': self._obs(self.obs_next)}

    def close(self):
        pass


class SyntheticMixedEnv:
    """Batched device-resident env with MIXED observations: one uint8 camera frame [C, H, W] and low-dim inputs per actor (the
    robosuite observation, ppo_configs.py:111-114).  The frame follows SyntheticPixelEnv (fresh uniform random bytes every
    step); the low-dim state follows SyntheticEnv (s' = tanh(Ws s + Wa a) + 0.01 xi); reward and done follow SyntheticEnv
    (r = -|s|^2 / D + 0.1 xi', done at ``limit_episode_length``).  One kernel per step writes every actor's observation
    straight into its packed record row (utils.obs_layout), which the window-staging kernels copy as opaque words; ``obs``
    hands out views into those rows: ``'pixel'/'camera0'`` and one view per low-dim key."""
    metadata = {}
    graph_safe = True

    def __init__(self, num_envs, obs_spec, action_dim=8, limit_episode_length=200, seed=0, device=None):
        from ..utils import obs_layout, obs_is_mixed
        if not torch.cuda.is_available():
            raise RuntimeError('SyntheticMixedEnv is device-resident: a CUDA device is required')
        if not obs_is_mixed(obs_spec):
            raise ValueError('SyntheticMixedEnv needs a spec with a camera frame and low-dim inputs, got %s' % (obs_spec,))
        self.device = torch.device(device if device is not None else ('cuda:%d' % torch.cuda.current_device()))
        self.spec = {'pixel': {'camera0': tuple(obs_spec['pixel']['camera0'])},
                     'low_dim': {k: tuple(v) for k, v in obs_spec['low_dim'].items()}}
        self.layout = obs_layout(self.spec)
        self.N, self.A = num_envs, action_dim
        self.D = self.layout['width']                 # words per packed row: what the staging / replay records carry
        self.low_dim = self.layout['low_dim']
        self.max_steps = int(limit_episode_length)
        self.seed = int(seed)
        Dl = self.low_dim
        g = torch.Generator().manual_seed(self.seed)  # as SyntheticEnv: the same seed gives the same low-dim dynamics
        scale = 1.0 / (Dl ** 0.5)
        self.Ws = (torch.randn(Dl, Dl, generator=g) * scale).to(self.device)
        self.Wa = (torch.randn(Dl, action_dim, generator=g) * scale).to(self.device)
        self.WsT, self.WaT = self.Ws.t().contiguous(), self.Wa.t().contiguous()
        self._g = torch.Generator().manual_seed(self.seed + 1)
        self.state = torch.zeros(num_envs, self.D, device=self.device)      # packed rows the actors observe next
        self.obs_next = torch.zeros_like(self.state)                         # true successors (terminal where done)
        self.ep_step = torch.zeros(num_envs, dtype=torch.int32, device=self.device)
        self.reward = torch.zeros(num_envs, device=self.device)
        self.done = torch.zeros(num_envs, device=self.device)
        self.step_counter = torch.zeros(1, dtype=torch.int64, device=self.device)
        from ..utils import mixed_obs_views
        self._obs_state, self._obs_next = mixed_obs_views(self.state, self.layout), mixed_obs_views(self.obs_next, self.layout)

    def observation_spec(self):
        return self.spec

    def action_spec(self):
        return {'dim': (self.A,), 'type': 'continuous'}

    def reset(self):
        lay, N = self.layout, self.N
        off = lay['low_dim_off']
        frames = torch.randint(0, 256, (N, lay['frame_bytes']), generator=self._g, dtype=torch.uint8)
        self.state.view(torch.uint8)[:, :lay['frame_bytes']].copy_(frames.to(self.device))
        self.state[:, off:off + self.low_dim].copy_(torch.randn(N, self.low_dim, generator=self._g).to(self.device))
        self.ep_step.zero_()
        return self._obs_state, {}

    def step(self, action):
        if isinstance(action, tuple):
            action = action[0]
        lay = self.layout
        check(_lib.lib().sb200_synth_mixed_env_step_f32(
            _p(self.state), _p(action), _p(self.WsT), _p(self.WaT), self.N, self.low_dim, self.A, lay['frame_bytes'] // 4,
            self.D, self.max_steps, _p(self.ep_step), self.seed + 7, _p(self.step_counter), _p(self.obs_next), _p(self.reward),
            _p(self.done), _stream()), 'sb200_synth_mixed_env_step_f32')
        return self._obs_state, self.reward, self.done, {'obs_next': self._obs_next}

    def close(self):
        pass
