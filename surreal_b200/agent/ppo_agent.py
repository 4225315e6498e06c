"""PPOAgent: drop-in for surreal/agent/ppo_agent.py:15-190 serving a whole batch of actors per call.

``act(obs)`` runs the fused actor MLP for all N actors in one launch, then one sampling kernel that
applies each actor's constant exploration scale exp(noise_i) (drawn once, ppo_agent.py:57-61), samples
N(mean, std), clips to [-1, 1] and records the behaviour policy AFTER scaling (ppo_agent.py:139,149).
numpy observations (a single actor's [D] vector or an [N, D] batch) are accepted for external CPU envs."""
import ctypes as C
import time

import numpy as np
import torch

from .. import _lib, ops
from .._lib import check
from ..model.ppo_net import PPOModel, DiagGauss
from ..env import ExpSenderWrapperMultiStepMovingWindowWithInfo
from .base import Agent


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class PPOAgent(Agent):
    def __init__(self, learner_config, env_config, session_config, agent_id, agent_mode, render=False):
        super().__init__(learner_config=learner_config, env_config=env_config, session_config=session_config,
                         agent_id=agent_id, agent_mode=agent_mode, render=render)
        if not torch.cuda.is_available():
            raise RuntimeError('surreal_b200.PPOAgent needs a CUDA device (there is no CPU fallback)')
        self.device = torch.device('cuda', torch.cuda.current_device())
        self.action_dim = self.env_config.action_spec.dim[0]
        self.obs_spec = self.env_config.obs_spec
        self.use_z_filter = self.learner_config.algo.use_z_filter
        self.init_log_sig = self.learner_config.algo.consts.init_log_sig
        self.log_sig_range = self.learner_config.algo.consts.log_sig_range
        if self.agent_mode != 'training':
            if self.agent_mode not in ['eval_deterministic_local', 'eval_stochastic_local']:
                self.agent_mode = 'eval_stochastic' if self.env_config.stochastic_eval else 'eval_deterministic'
        N = self.num_envs
        if self.agent_mode != 'training':
            self.noise = np.zeros(N)
        else:                                  # one constant per actor (ppo_agent.py:60-61)
            self.noise = np.random.uniform(low=-self.log_sig_range, high=self.log_sig_range, size=N)
        self.rnn_config = self.learner_config.algo.rnn
        self.gpu_ids = 'cuda:all'
        self.pd = DiagGauss(self.action_dim)
        self.cells = None
        pixel = bool(self.env_config.pixel_input) if 'pixel_input' in self.env_config else False
        self.model = PPOModel(obs_spec=self.obs_spec, action_dim=self.action_dim, model_config=self.learner_config.model,
                              use_cuda=True, init_log_sig=self.init_log_sig, use_z_filter=self.use_z_filter,
                              if_pixel_input=pixel, rnn_config=self.rnn_config, device=self.device)
        A, D = self.action_dim, self.model.low_dim
        self._log_noise = torch.tensor(self.noise, dtype=torch.float32, device=self.device)
        self._mean = torch.zeros(N, A, device=self.device)
        self._packed = ops.PackedWeights(self.model.actor)          # per-step inference copy of the policy weights
        self._action = torch.zeros(N, A, device=self.device)
        self._pd = torch.zeros(N, 2 * A, device=self.device)
        self._obs_dev = torch.zeros(N, D, device=self.device)
        self._obs_pin = None
        self._out_pin = None
        self._counter = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.seed = 2 + 1000003 * int(agent_id)

    def set_noise(self, noise):
        self.noise = np.asarray(noise, dtype=np.float64).reshape(self.num_envs)
        self._log_noise.copy_(torch.tensor(self.noise, dtype=torch.float32))

    def act(self, obs, eps=None):
        """-> action (eval) or (action, [onetime_infos, [pd]]) in training, like ppo_agent.py:151-154.
        Device observations give device results; numpy in, numpy out."""
        N, A, D = self.num_envs, self.action_dim, self.model.low_dim
        if self.model.mixed:
            return self._act_mixed(obs, eps)
        if self.model.cnn_stem is not None:
            return self._act_pixel(obs, eps)
        if self.model.rnn_stem is not None:
            return self._act_rnn(obs, eps)
        x = obs
        if isinstance(obs, dict):
            xs = [obs['low_dim'][k] for k in obs['low_dim']]
            x = xs[0] if len(xs) == 1 else (torch.cat(xs, -1) if isinstance(xs[0], torch.Tensor)
                                            else np.concatenate(xs, -1))
        host = not isinstance(x, torch.Tensor)
        if host and eps is None and isinstance(x, np.ndarray):
            return self._act_host(obs, x)                          # one C call: copies, kernels, one sync
        if host:
            cached = self.env.cached_device_obs(x) if hasattr(self.env, 'cached_device_obs') else None
            if cached is not None:
                x = cached                                         # the wrapper already moved this observation
            else:
                if self._obs_pin is None:
                    self._obs_pin = torch.empty(N, D, dtype=torch.float32, pin_memory=True)
                xt = torch.from_numpy(x) if (isinstance(x, np.ndarray) and x.dtype == np.float32 and
                                             x.flags['C_CONTIGUOUS'] and x.flags['WRITEABLE']) else None
                if xt is not None and xt.is_pinned():              # observation already in pinned memory: DMA directly
                    self._obs_dev.copy_(xt.view(N, D), non_blocking=True)
                else:
                    self._obs_pin.numpy()[...] = np.asarray(x, dtype=np.float32).reshape(N, D)
                    self._obs_dev.copy_(self._obs_pin, non_blocking=True)
                x = self._obs_dev
        x = x.reshape(N, D)
        m = self.model
        if self._in_chunk and self._packed.supported and x.stride(1) == 1:
            # inside a multi-step chunk the weights are fixed: the chunk packed them once, at its top
            ops.mlp_forward_packed(self._packed, x, zf_stats=m.z_stats, zf_eps=m.z_eps, out=self._mean)
        else:
            ops.mlp_forward(m.actor, x, zf_stats=m.z_stats, zf_eps=m.z_eps, out=self._mean)
        det = self.agent_mode in ['eval_deterministic', 'eval_deterministic_local']
        env = self.env
        staged = self.agent_mode == 'training' and isinstance(env, ExpSenderWrapperMultiStepMovingWindowWithInfo)
        counter = env.step_counter if (env is not None and hasattr(env, 'step_counter')) else self._counter
        eps_dev = None
        if eps is not None:
            eps_dev = torch.as_tensor(np.asarray(eps, dtype=np.float32).reshape(N, A)).to(self.device)
        if staged and counter is not self._counter and env.fuse_launches:
            # sampling + this step's replay-slot assignment + step-counter advance in one launch
            fifo_state, dest = env.slot_assignment_args()
            check(_lib.lib().sb200_ppo_sample_assign_f32(
                _p(self._mean), A, _p(m.log_var), _p(self._log_noise), _p(eps_dev), N, A, int(det), self.seed,
                _p(counter), _p(self._action), _p(self._pd), _p(env.stage_pos), _p(env.stage_act), _p(env.stage_pd),
                env.n_step, _p(fifo_state), _p(dest), ops._stream()), 'sb200_ppo_sample_assign_f32')
        else:
            check(_lib.lib().sb200_ppo_sample_f32(
                _p(self._mean), A, _p(m.log_var), _p(self._log_noise), _p(eps_dev), N, A, int(det), self.seed,
                _p(counter), _p(self._action), _p(self._pd), _p(env.stage_pos) if staged else None,
                _p(env.stage_act) if staged else None, _p(env.stage_pd) if staged else None,
                env.n_step if staged else 1, ops._stream()), 'sb200_ppo_sample_f32')
        if not staged and counter is self._counter:
            self._counter += 1
        if host:
            if self._out_pin is None:
                self._out_pin = (torch.empty(N, A, dtype=torch.float32, pin_memory=True),
                                 torch.empty(N, 2 * A, dtype=torch.float32, pin_memory=True))
            self._out_pin[0].copy_(self._action, non_blocking=True)
            self._out_pin[1].copy_(self._pd, non_blocking=True)
            torch.cuda.current_stream().synchronize()              # one sync for both D2H copies
            action = self._out_pin[0].numpy().astype(np.float64)   # the reference hands the env float64 (ppo_net.py:83)
            pd = self._out_pin[1].numpy().copy()
            if N == 1 and np.asarray(obs['low_dim'][next(iter(obs['low_dim']))] if isinstance(obs, dict) else obs).ndim == 1:
                action, pd = action.reshape(-1), pd.reshape(-1)
        else:
            action, pd = self._action, self._pd
        if self.agent_mode != 'training':
            return action
        if self.env_config.sleep_time:
            time.sleep(self.env_config.sleep_time)
        return action, [[], [pd]]

    # -- RNN policy (the reference's default PPO config) ------------------------------------------------------------
    def _rnn_state(self):
        """LSTM cells of all N actors, zero-initialised (ppo_agent.py:84-93).  NOTE: like the reference -- whose
        ``reset()`` no caller ever invokes -- the cells carry over from episode to episode."""
        if getattr(self, '_h', None) is None:
            N, H, D = self.num_envs, self.model.rnn_stem.H, self.model.low_dim
            z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=self.device)  # noqa: E731
            self._h, self._c, self._h_before, self._c_before = z(N, H), z(N, H), z(N, H), z(N, H)
            self._xf = z(N, ops._ru(D, 4))[:, :D]
            self._rnn_bufs = self.model.rnn_stem.buffers(N, 1, save=False)
            self._aug_bufs = [z(N, D + 2 * H), z(N, D + 2 * H)]
        return self._h, self._c

    def _augment(self, o, which=0):
        """Observation rows + the cells this agent holds right now (what it will act FROM on that observation): the rows the
        HBM staging / replay carry in RNN mode (utils.record_obs_dim)."""
        h, c = self._rnn_state()
        D, H = self.model.low_dim, self.model.rnn_stem.H
        buf = self._aug_bufs[which]
        buf[:, :D].copy_(o.reshape(self.num_envs, D), non_blocking=True)
        buf[:, D:D + H].copy_(h, non_blocking=True)
        buf[:, D + H:].copy_(c, non_blocking=True)
        return buf

    def _act_rnn(self, obs, eps=None):
        """act() with the LSTM stem: z-filter -> one LSTM step from each actor's cells -> actor head -> sampling
        (ppo_net.py:317-351, ppo_agent.py:133-149).  The cells BEFORE the step are the step's onetime_info."""
        from ..model.lstm_stem import rows_zfilter
        N, A, D = self.num_envs, self.action_dim, self.model.low_dim
        m, stem = self.model, self.model.rnn_stem
        h, c = self._rnn_state()
        x = obs
        if isinstance(obs, dict):
            xs = [obs['low_dim'][k] for k in obs['low_dim']]
            x = xs[0] if len(xs) == 1 else (torch.cat(xs, -1) if isinstance(xs[0], torch.Tensor) else np.concatenate(xs, -1))
        host = not isinstance(x, torch.Tensor)
        if host:
            if self._obs_pin is None:
                self._obs_pin = torch.empty(N, D, dtype=torch.float32, pin_memory=True)
            self._obs_pin.numpy()[...] = np.asarray(x, dtype=np.float32).reshape(N, D)
            self._obs_dev.copy_(self._obs_pin, non_blocking=True)
            x = self._obs_dev
        x = x.reshape(N, D)
        self._h_before.copy_(h, non_blocking=True)
        self._c_before.copy_(c, non_blocking=True)
        rows_zfilter(x, D, x.stride(0), N, 1, D, m.z_stats, m.z_eps, self._xf)
        feat = stem.forward(self._xf, h, c, h.stride(0), N, 1, self._rnn_bufs, h_last=h, c_last=c)     # cells updated in place
        ops.mlp_forward(m.actor, feat, out=self._mean)
        det = self.agent_mode in ['eval_deterministic', 'eval_deterministic_local']
        env = self.env
        staged = self.agent_mode == 'training' and isinstance(env, ExpSenderWrapperMultiStepMovingWindowWithInfo)
        counter = env.step_counter if (env is not None and hasattr(env, 'step_counter')) else self._counter
        eps_dev = None
        if eps is not None:
            eps_dev = torch.as_tensor(np.asarray(eps, dtype=np.float32).reshape(N, A)).to(self.device)
        if staged and counter is not self._counter and env.fuse_launches:
            fifo_state, dest = env.slot_assignment_args()
            check(_lib.lib().sb200_ppo_sample_assign_f32(
                _p(self._mean), A, _p(m.log_var), _p(self._log_noise), _p(eps_dev), N, A, int(det), self.seed,
                _p(counter), _p(self._action), _p(self._pd), _p(env.stage_pos), _p(env.stage_act), _p(env.stage_pd),
                env.n_step, _p(fifo_state), _p(dest), ops._stream()), 'sb200_ppo_sample_assign_f32')
        else:
            check(_lib.lib().sb200_ppo_sample_f32(
                _p(self._mean), A, _p(m.log_var), _p(self._log_noise), _p(eps_dev), N, A, int(det), self.seed,
                _p(counter), _p(self._action), _p(self._pd), _p(env.stage_pos) if staged else None,
                _p(env.stage_act) if staged else None, _p(env.stage_pd) if staged else None,
                env.n_step if staged else 1, ops._stream()), 'sb200_ppo_sample_f32')
        if not staged and counter is self._counter:
            self._counter += 1
        if host:
            torch.cuda.current_stream().synchronize()
            action = self._action.cpu().numpy().astype(np.float64)
            pd = self._pd.cpu().numpy()
            onetime = [self._h_before.cpu().numpy()[:, None, :], self._c_before.cpu().numpy()[:, None, :]]   # [N, layers, H]
            if N == 1:
                action, pd, onetime = action.reshape(-1), pd.reshape(-1), [onetime[0][0], onetime[1][0]]
        else:
            action, pd = self._action, self._pd
            onetime = [self._h_before.unsqueeze(1), self._c_before.unsqueeze(1)]
        if self.agent_mode != 'training':
            return action
        if self.env_config.sleep_time:
            time.sleep(self.env_config.sleep_time)
        return action, [onetime, [pd]]

    def _act_pixel(self, obs, eps=None):
        """act() on uint8 frames [N, C, H, W] (device tensor or numpy): CNN stem -> actor head -> sampling kernel
        (ppo_net.py:268-273,368-375; ppo_agent.py:138-149)."""
        N, A = self.num_envs, self.action_dim
        m, stem = self.model, self.model.cnn_stem
        fr = obs['pixel']['camera0'] if isinstance(obs, dict) else obs
        host = not isinstance(fr, torch.Tensor)
        if host:
            if self._obs_pin is None:
                self._obs_pin = torch.empty(N, stem.C, stem.H, stem.W, dtype=torch.uint8, pin_memory=True)
                self._frames_dev = torch.empty(N, stem.C, stem.H, stem.W, dtype=torch.uint8, device=self.device)
            self._obs_pin.numpy()[...] = np.asarray(fr, dtype=np.uint8).reshape(N, stem.C, stem.H, stem.W)
            self._frames_dev.copy_(self._obs_pin, non_blocking=True)
            fr = self._frames_dev
        fr = fr.reshape(N, stem.C, stem.H, stem.W)
        if getattr(self, '_stem_bufs', None) is None:
            self._stem_bufs = stem.buffers(N)
        feat = stem.forward(fr, self._stem_bufs)
        ops.mlp_forward(m.actor, feat, out=self._mean)
        det = self.agent_mode in ['eval_deterministic', 'eval_deterministic_local']
        env = self.env
        staged = self.agent_mode == 'training' and isinstance(env, ExpSenderWrapperMultiStepMovingWindowWithInfo)
        counter = env.step_counter if (env is not None and hasattr(env, 'step_counter')) else self._counter
        eps_dev = None
        if eps is not None:
            eps_dev = torch.as_tensor(np.asarray(eps, dtype=np.float32).reshape(N, A)).to(self.device)
        if staged and counter is not self._counter and env.fuse_launches:
            fifo_state, dest = env.slot_assignment_args()
            check(_lib.lib().sb200_ppo_sample_assign_f32(
                _p(self._mean), A, _p(m.log_var), _p(self._log_noise), _p(eps_dev), N, A, int(det), self.seed,
                _p(counter), _p(self._action), _p(self._pd), _p(env.stage_pos), _p(env.stage_act), _p(env.stage_pd),
                env.n_step, _p(fifo_state), _p(dest), ops._stream()), 'sb200_ppo_sample_assign_f32')
        else:
            check(_lib.lib().sb200_ppo_sample_f32(
                _p(self._mean), A, _p(m.log_var), _p(self._log_noise), _p(eps_dev), N, A, int(det), self.seed,
                _p(counter), _p(self._action), _p(self._pd), _p(env.stage_pos) if staged else None,
                _p(env.stage_act) if staged else None, _p(env.stage_pd) if staged else None,
                env.n_step if staged else 1, ops._stream()), 'sb200_ppo_sample_f32')
        if not staged and counter is self._counter:
            self._counter += 1
        if host:
            if self._out_pin is None:
                self._out_pin = (torch.empty(N, A, dtype=torch.float32, pin_memory=True),
                                 torch.empty(N, 2 * A, dtype=torch.float32, pin_memory=True))
            self._out_pin[0].copy_(self._action, non_blocking=True)
            self._out_pin[1].copy_(self._pd, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            action, pd = self._out_pin[0].numpy().astype(np.float64), self._out_pin[1].numpy().copy()
        else:
            action, pd = self._action, self._pd
        if self.agent_mode != 'training':
            return action
        if self.env_config.sleep_time:
            time.sleep(self.env_config.sleep_time)
        return action, [[], [pd]]

    def _act_mixed(self, obs, eps=None):
        """act() on mixed observations (a camera frame + low-dim inputs): CNN stem on the frames -> actor head on
        cat(zfilter(low_dim), features) (ppo_net.py:262-275) -> sampling kernel.  Both parts are read in place from the
        packed observation rows (utils.obs_layout): the device env's own rows, or a host dict packed into a pinned row."""
        from ..utils import obs_flat, obs_layout, pack_obs_rows
        N, A = self.num_envs, self.action_dim
        m, stem = self.model, self.model.cnn_stem
        if getattr(self, '_layout', None) is None:
            self._layout = obs_layout(self.obs_spec)
            self._stem_bufs = stem.buffers(N)
        lay = self._layout
        W = lay['width']
        host = not isinstance(obs['pixel']['camera0'], torch.Tensor)
        if host:
            if self._obs_pin is None:
                self._obs_pin = torch.zeros(N, W, dtype=torch.float32, pin_memory=True)
                self._rows_dev = torch.zeros(N, W, dtype=torch.float32, device=self.device)
            pack_obs_rows(obs, lay, out=self._obs_pin.numpy())
            self._rows_dev.copy_(self._obs_pin, non_blocking=True)
            rows = self._rows_dev
        else:
            rows = obs_flat(obs, self.obs_spec)
        feat = stem.forward(rows, self._stem_bufs, rows=N, row_bytes=4 * W)
        ops.mlp_forward(m.actor, rows[:, lay['low_dim_off']:], zf_stats=m.z_stats, zf_eps=m.z_eps, aux=feat, rows=N, ldx=W,
                        out=self._mean)
        return self._sample(eps, host)

    def _sample(self, eps, host):
        """Sampling kernel on self._mean (+ staging of action / pd rows in training), then the act() return value."""
        N, A, m = self.num_envs, self.action_dim, self.model
        det = self.agent_mode in ['eval_deterministic', 'eval_deterministic_local']
        env = self.env
        staged = self.agent_mode == 'training' and isinstance(env, ExpSenderWrapperMultiStepMovingWindowWithInfo)
        counter = env.step_counter if (env is not None and hasattr(env, 'step_counter')) else self._counter
        eps_dev = None
        if eps is not None:
            eps_dev = torch.as_tensor(np.asarray(eps, dtype=np.float32).reshape(N, A)).to(self.device)
        if staged and counter is not self._counter and env.fuse_launches:
            fifo_state, dest = env.slot_assignment_args()
            check(_lib.lib().sb200_ppo_sample_assign_f32(
                _p(self._mean), A, _p(m.log_var), _p(self._log_noise), _p(eps_dev), N, A, int(det), self.seed,
                _p(counter), _p(self._action), _p(self._pd), _p(env.stage_pos), _p(env.stage_act), _p(env.stage_pd),
                env.n_step, _p(fifo_state), _p(dest), ops._stream()), 'sb200_ppo_sample_assign_f32')
        else:
            check(_lib.lib().sb200_ppo_sample_f32(
                _p(self._mean), A, _p(m.log_var), _p(self._log_noise), _p(eps_dev), N, A, int(det), self.seed,
                _p(counter), _p(self._action), _p(self._pd), _p(env.stage_pos) if staged else None,
                _p(env.stage_act) if staged else None, _p(env.stage_pd) if staged else None,
                env.n_step if staged else 1, ops._stream()), 'sb200_ppo_sample_f32')
        if not staged and counter is self._counter:
            self._counter += 1
        if host:
            if self._out_pin is None:
                self._out_pin = (torch.empty(N, A, dtype=torch.float32, pin_memory=True),
                                 torch.empty(N, 2 * A, dtype=torch.float32, pin_memory=True))
            self._out_pin[0].copy_(self._action, non_blocking=True)
            self._out_pin[1].copy_(self._pd, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            action, pd = self._out_pin[0].numpy().astype(np.float64), self._out_pin[1].numpy().copy()
        else:
            action, pd = self._action, self._pd
        if self.agent_mode != 'training':
            return action
        if self.env_config.sleep_time:
            time.sleep(self.env_config.sleep_time)
        return action, [[], [pd]]

    def _act_host(self, obs, x):
        """act() for a HOST observation batch through sb200_ppo_act_host_f32 (H2D -> forward -> sample -> D2H -> sync
        issued back to back from C): numpy in, numpy out, same results as the generic path."""
        N, A, D = self.num_envs, self.action_dim, self.model.low_dim
        m, env = self.model, self.env
        if self._out_pin is None:
            self._out_pin = (torch.empty(N, A, dtype=torch.float32, pin_memory=True),
                             torch.empty(N, 2 * A, dtype=torch.float32, pin_memory=True))
        cached = env.cached_device_obs(x) if hasattr(env, 'cached_device_obs') else None
        if cached is not None:
            obs_host, obs_dev = None, cached                       # the wrapper already moved this observation
        else:
            src = x if (x.dtype == np.float32 and x.flags['C_CONTIGUOUS'] and x.flags['WRITEABLE'] and
                        torch.from_numpy(x).is_pinned()) else None
            if src is None:
                if self._obs_pin is None:
                    self._obs_pin = torch.empty(N, D, dtype=torch.float32, pin_memory=True)
                self._obs_pin.numpy()[...] = np.asarray(x, dtype=np.float32).reshape(N, D)
                src = self._obs_pin.numpy()
            obs_host, obs_dev = C.c_void_p(src.ctypes.data), self._obs_dev
        det = self.agent_mode in ['eval_deterministic', 'eval_deterministic_local']
        staged = self.agent_mode == 'training' and isinstance(env, ExpSenderWrapperMultiStepMovingWindowWithInfo)
        counter = env.step_counter if (env is not None and hasattr(env, 'step_counter')) else self._counter
        fifo_state = dest = None
        if staged and counter is not self._counter and env.fuse_launches:
            fifo_state, dest = env.slot_assignment_args()
        d = m.actor.desc()
        zf = ops.zfilter_desc(m.z_stats, m.z_eps)
        check(_lib.lib().sb200_ppo_act_host_f32(
            C.byref(d), C.byref(zf), obs_host, _p(obs_dev), N, _p(self._mean), _p(m.log_var), _p(self._log_noise),
            int(det), self.seed, _p(counter), _p(self._action), _p(self._pd), _p(env.stage_pos) if staged else None,
            _p(env.stage_act) if staged else None, _p(env.stage_pd) if staged else None, env.n_step if staged else 1,
            _p(fifo_state), _p(dest), C.c_void_p(self._out_pin[0].data_ptr()), C.c_void_p(self._out_pin[1].data_ptr()),
            ops._stream()), 'sb200_ppo_act_host_f32')
        if not staged and counter is self._counter:
            self._counter += 1
        action = self._out_pin[0].numpy().astype(np.float64)       # the reference hands the env float64 (ppo_net.py:83)
        pd = self._out_pin[1].numpy().copy()
        o0 = obs['low_dim'][next(iter(obs['low_dim']))] if isinstance(obs, dict) else obs
        if N == 1 and np.asarray(o0).ndim == 1:
            action, pd = action.reshape(-1), pd.reshape(-1)
        if self.agent_mode != 'training':
            return action
        if self.env_config.sleep_time:
            time.sleep(self.env_config.sleep_time)
        return action, [[], [pd]]

    def rollout_chunk_supported(self):
        """True when ``steps`` consecutive act -> env.step -> staging iterations can run as the persistent rollout
        kernel (sb200_ppo_rollout_f32): training mode, the in-tree device env behind the window wrapper, and a policy
        that fits the kernel's shared-memory plan."""
        import os
        from ..env import SyntheticEnv
        env = self.env
        if self.agent_mode != 'training' or os.environ.get('SB200_PERSISTENT_ROLLOUT', '1') == '0':
            return False
        if self.model.rnn_stem is not None or self.model.cnn_stem is not None:
            return False                       # the persistent kernel runs the plain MLP policy only
        if not isinstance(env, ExpSenderWrapperMultiStepMovingWindowWithInfo) or not env.persistent_rollout:
            return False
        if type(env.env) is not SyntheticEnv:
            return False
        d = self.model.actor.desc()
        return bool(_lib.lib().sb200_ppo_rollout_supported(C.byref(d), self.model.low_dim, self.action_dim))

    def rollout_chunk(self, steps):
        """``steps`` iterations of the actor loop (agent/base.py:244-262) in one launch + the ordered commit pass."""
        w = self.env
        e, r, m = w.env, w.replay, self.model
        ob = w.rollout_outbox(steps)
        if ob is None:
            return False
        a = _lib.PPORollout()
        d = m.actor.desc()
        a.net = C.pointer(d)
        a.zf_stats = m.z_stats.data_ptr() if m.z_stats is not None else None
        a.zf_eps = float(m.z_eps)
        a.log_var, a.log_noise = m.log_var.data_ptr(), self._log_noise.data_ptr()
        a.agent_seed, a.deterministic = self.seed, 0
        a.state, a.WsT, a.WaT, a.ep_step = e.state.data_ptr(), e.WsT.data_ptr(), e.WaT.data_ptr(), e.ep_step.data_ptr()
        a.max_steps, a.env_seed = e.max_steps, e.seed + 7
        a.action, a.pd = self._action.data_ptr(), self._pd.data_ptr()
        a.obs_next, a.reward, a.done = e.obs_next.data_ptr(), e.reward.data_ptr(), e.done.data_ptr()
        a.stage_pos, a.stage_obs, a.stage_act = w.stage_pos.data_ptr(), w.stage_obs.data_ptr(), w.stage_act.data_ptr()
        a.stage_pd, a.stage_rew, a.stage_done = w.stage_pd.data_ptr(), w.stage_rew.data_ptr(), w.stage_done.data_ptr()
        a.o_obs, a.o_act, a.o_pd = ob['o_obs'].data_ptr(), ob['o_act'].data_ptr(), ob['o_pd'].data_ptr()
        a.o_rew, a.o_done = ob['o_rew'].data_ptr(), ob['o_done'].data_ptr()
        a.ev_step, a.ev_count, a.W = ob['ev_step'].data_ptr(), ob['ev_count'].data_ptr(), ob['W']
        a.N, a.D, a.A = self.num_envs, m.low_dim, self.action_dim
        a.n_step, a.stride, a.T = w.n_step, w.stride, int(steps)
        a.step_counter = e.step_counter.data_ptr()
        L, st = _lib.lib(), ops._stream()
        check(L.sb200_ppo_rollout_f32(C.byref(a), st), 'sb200_ppo_rollout_f32')
        check(L.sb200_ppo_rollout_commit_f32(C.byref(a), _p(ob['scratch']), _p(r.state), _p(r.r_obs), _p(r.r_act),
                                             _p(r.r_pd), _p(r.r_rew), _p(r.r_done), _p(e.step_counter), st),
              'sb200_ppo_rollout_commit_f32')
        return True

    def module_dict(self):
        return {'ppo': self.model}

    def default_config(self):
        return {'model': {'convs': '_list_', 'fc_hidden_sizes': '_list_'}}

    def reset(self):
        """reset of LSTM hidden and cell states (ppo_agent.py:169-183; nothing in the reference calls it)."""
        if self.model.rnn_stem is not None and getattr(self, '_h', None) is not None:
            self._h.zero_()
            self._c.zero_()

    def prepare_env_agent(self, env):
        env = super().prepare_env_agent(env)
        if self.model.rnn_stem is not None:
            self._rnn_state()
            w = ExpSenderWrapperMultiStepMovingWindowWithInfo(env, self.learner_config, self.session_config,
                                                              obs_extra=2 * self.model.rnn_stem.H)
            w.obs_augment = self._augment
            w.persistent_rollout = False
            return w
        return ExpSenderWrapperMultiStepMovingWindowWithInfo(env, self.learner_config, self.session_config)
