"""PPOLearner: drop-in for surreal/learner/ppo.py:12-682 whose learn() runs entirely as hand-written
sm_100a kernels (critic pass -> windowed GAE -> fused loss+grad -> backward GEMMs -> clip+Adam).

Same constructor, config keys, method names, statistics names and control flow as the reference
(clip / adapt modes, KL early stop ppo.py:556, publish-time adaptation ppo.py:637-666).  The batch a
``learn(batch)`` call receives has the aggregator's layout (aggregator.py:176-183); its arrays may be
numpy (copied through pinned memory) or CUDA tensors (zero copy).
"""
import ctypes as C
import os

import numpy as np
import torch

from .. import _lib, ops
from .. import utils as U
from .._lib import check
from ..model.ppo_net import PPOModel, DiagGauss
from ..session import ConfigError
from .aggregator import MultistepAggregatorWithInfo
from .base import Learner
from .scheduler import make_lr_scheduler

S = dict(SURR=0, LOSS=1, ENTROPY=2, KL_PRE=3, KL_POST=4, GN_ACTOR=5, VAL_LOSS=6, EXPL_VAR=7, GN_CRITIC=8,
         RET_MEAN=9, LOG_SIG=10, BEHAVE_LIK=11, IS_WEIGHT=12, REF_BEHAVE=13, EPOCHS=14, VAL_MOMENTS=16, COUNT=32)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def stem_shape(stem):
    return (stem.C, stem.H, stem.W)


class PPOLearner(Learner):
    def __init__(self, learner_config, env_config, session_config):
        super().__init__(learner_config, env_config, session_config)
        if not torch.cuda.is_available():
            raise RuntimeError('surreal_b200.PPOLearner needs a CUDA device (there is no CPU fallback)')
        self.device = torch.device('cuda', torch.cuda.current_device())
        self.gpu_option = 'cuda:all'
        self.use_cuda = True
        self.current_iteration = 0
        self.global_step = 0
        lc = self.learner_config

        # RL general parameters (ppo.py:75-85)
        self.gamma = lc.algo.gamma
        self.lam = lc.algo.advantage.lam
        self.n_step = lc.algo.n_step
        self.use_z_filter = lc.algo.use_z_filter
        self.use_r_filter = lc.algo.use_r_filter
        self.norm_adv = lc.algo.advantage.norm_adv
        self.batch_size = lc.replay.batch_size
        self.action_dim = self.env_config.action_spec.dim[0]
        self.obs_spec = self.env_config.obs_spec
        self.init_log_sig = lc.algo.consts.init_log_sig

        # PPO parameters (ppo.py:88-118)
        self.ppo_mode = lc.algo.ppo_mode
        if self.ppo_mode not in ('adapt', 'clip'):
            raise ConfigError('ppo_mode must be "adapt" or "clip"')
        self.if_rnn_policy = lc.algo.rnn.if_rnn_policy
        self.horizon = lc.algo.rnn.horizon
        self.lr_actor = lc.algo.network.lr_actor
        self.lr_critic = lc.algo.network.lr_critic
        self.epoch_policy = lc.algo.consts.epoch_policy
        self.epoch_baseline = lc.algo.consts.epoch_baseline
        self.kl_target = lc.algo.consts.kl_target
        self.adjust_threshold = lc.algo.consts.adjust_threshold
        self.reward_scale = lc.algo.advantage.reward_scale
        self.kl_cutoff_coeff = lc.algo.adapt_consts.kl_cutoff_coeff
        self.beta_init = lc.algo.adapt_consts.beta_init
        self.beta_range = lc.algo.adapt_consts.beta_range
        self.clip_range = lc.algo.clip_consts.clip_range
        self.clip_epsilon_init = lc.algo.clip_consts.clip_epsilon_init
        if self.ppo_mode == 'adapt':
            self.beta = self.beta_init
            self.eta = self.kl_cutoff_coeff
            self.beta_upper, self.beta_lower = self.beta_range[1], self.beta_range[0]
            self.beta_adjust_threshold = self.adjust_threshold
        else:
            self.clip_epsilon = self.clip_epsilon_init
            self.clip_adjust_threshold = self.adjust_threshold
            self.clip_upper, self.clip_lower = self.clip_range[1], self.clip_range[0]
            self.eta = self.kl_cutoff_coeff

        self.exp_counter = 0
        self.kl_record = []

        pixel = bool(self.env_config.pixel_input) if 'pixel_input' in self.env_config else False
        mk = dict(obs_spec=self.obs_spec, action_dim=self.action_dim, model_config=lc.model, use_cuda=True,
                  init_log_sig=self.init_log_sig, use_z_filter=self.use_z_filter, if_pixel_input=pixel,
                  rnn_config=lc.algo.rnn, device=self.device)
        self.model = PPOModel(**mk)
        self.ref_target_model = PPOModel(**mk)
        self.ref_target_model.update_target_params(self.model)

        net = lc.algo.network
        self.clip_actor_gradient = net.clip_actor_gradient
        self.actor_gradient_clip_value = net.actor_gradient_norm_clip
        self.clip_critic_gradient = net.clip_critic_gradient
        self.critic_gradient_clip_value = net.critic_gradient_norm_clip

        B, n, A = self.batch_size, self.n_step, self.action_dim
        self.pixel = self.model.cnn_stem is not None
        # mixed observations (frame + low-dim): the pixel-mode launch chain with the low-dim columns as the heads' input and the
        # CNN features as their layer-0 aux input; both read in place from the record rows (utils.obs_layout)
        self.mixed = self.model.mixed
        self.obs_layout = U.obs_layout(self.obs_spec) if self.mixed else None
        self.rnn = self.model.rnn_stem is not None
        self.obs_dim = self.model.low_dim                         # width of the low-dim features themselves
        # width of one observation in the batch buffers: the low-dim features (+ the actor's LSTM cells h | c in RNN mode,
        # which ride in the observation rows of the HBM records -- the reference ships them as onetime_infos), or the uint8
        # frame as 32-bit words
        D = U.record_obs_dim(lc, self.env_config)
        self.low_dim = D
        self.eff_len = (n - self.horizon + 1) if self.rnn else 1
        M = B * self.eff_len                                      # rows the heads train on (ppo.py:518-537)
        self._rows = M
        dev = self.device
        ig = 'linear' if self.rnn else ('aux' if self.mixed else self.pixel)
        self.actor_optim = ops.MlpTrainer(self.model.actor, M, self.lr_actor,
                                          clip_mode=1 if self.clip_actor_gradient else 0,
                                          clip_value=self.actor_gradient_clip_value,
                                          weight_decay=net.actor_regularization, input_grad=ig)
        self.critic_optim = ops.MlpTrainer(self.model.critic, M, self.lr_critic,
                                           clip_mode=1 if self.clip_critic_gradient else 0,
                                           clip_value=self.critic_gradient_clip_value,
                                           weight_decay=net.critic_regularization, input_grad=ig)
        if self.rnn:
            # the LSTM stem is shared by actor and critic and trained by BOTH optimisers (ppo_net.py:202-224)
            from ..model.lstm_stem import RnnTrainer
            stem, E, Hh, od = self.model.rnn_stem, self.eff_len, self.model.rnn_stem.H, self.obs_dim
            self.actor_rnn, self.critic_rnn = RnnTrainer(stem, B, E), RnnTrainer(stem, B, E)
            self._g_actor = torch.zeros(self.model.actor.size + stem.size, dtype=torch.float32, device=dev)
            self._g_critic = torch.zeros(self.model.critic.size + stem.size, dtype=torch.float32, device=dev)
            self.actor_optim.grad = self._g_actor[:self.model.actor.size]
            self.critic_optim.grad = self._g_critic[:self.model.critic.size]
            zz = lambda r, w: torch.zeros(r, ops._ru(w, 4), dtype=torch.float32, device=dev)[:, :w]  # noqa: E731
            self._xf_all, self._xf_eff, self._xf_ref, self._xraw_eff = zz(B * (n + 1), od), zz(M, od), zz(M, od), zz(M, od)
            self._act_it, self._pd_it = torch.zeros(M, A, device=dev), torch.zeros(M, 2 * A, device=dev)
            self._rnn_all = stem.buffers(B, n + 1, save=False)
            self._rnn_ref = self.ref_target_model.rnn_stem.buffers(B, E, save=False)
        if self.pixel:
            # the CNN stem is shared by actor and critic and trained by BOTH optimisers, each with its own Adam state
            # (ppo_net.py:202-224): one StemTrainer per optimiser, gradients of head + stem in one contiguous buffer
            from ..model.cnn_stem import StemTrainer
            stem = self.model.cnn_stem
            self.actor_stem, self.critic_stem = StemTrainer(stem, B), StemTrainer(stem, B)
            self._g_actor = torch.zeros(self.model.actor.size + stem.size, dtype=torch.float32, device=dev)
            self._g_critic = torch.zeros(self.model.critic.size + stem.size, dtype=torch.float32, device=dev)
            self.actor_optim.grad = self._g_actor[:self.model.actor.size]
            self.critic_optim.grad = self._g_critic[:self.model.critic.size]
            # step-0 frames of every window, contiguous (pixel mode; mixed mode reads them in place)
            self._frames0 = None if self.mixed else torch.zeros(B, *stem_shape(stem), dtype=torch.uint8, device=dev)
            self._stem_all = None                                 # activation buffers of the B*(n+1)-frame critic pass
            self._ref_stem_bufs = self.ref_target_model.cnn_stem.buffers(B)

        # learning-rate schedule (ppo.py:121-125,171-178)
        an = net.anneal
        num_updates = int(an.frames_to_anneal / lc.parameter_publish.exp_interval)
        self.actor_lr_scheduler = make_lr_scheduler(an.lr_scheduler, self.actor_optim, self.lr_actor, num_updates,
                                                    update_freq=an.lr_update_frequency, min_lr=an.min_lr)
        self.critic_lr_scheduler = make_lr_scheduler(an.lr_scheduler, self.critic_optim, self.lr_critic, num_updates,
                                                     update_freq=an.lr_update_frequency, min_lr=an.min_lr)

        self.aggregator = MultistepAggregatorWithInfo(self.env_config.obs_spec, self.env_config.action_spec)
        self.pd = DiagGauss(self.action_dim)
        self.cells = None

        # ---- device state of one learn(): allocated once, reused (graph-friendly, no allocator traffic)
        f = lambda *sh: torch.zeros(*sh, dtype=torch.float32, device=dev)  # noqa: E731
        # own batch buffers (host-batch path); a device batch from the HBM replay is used in place instead
        self._own = dict(obs_full=f(B, n + 1, D), actions=f(B, n, A), pds=f(B, n, 2 * A), rewards=f(B, n),
                         dones=f(B, n))
        self._obs_full, self._actions, self._pds = self._own['obs_full'], self._own['actions'], self._own['pds']
        self._rewards, self._dones = self._own['rewards'], self._own['dones']
        self._rewards_f = f(B, n) if self.use_r_filter else None
        self._values = f(B * (n + 1), 1)
        self._adv, self._ret = f(B, self.eff_len), f(B, self.eff_len)
        self._ref_mean, self._ref_pd = f(M, A), f(M, 2 * A)
        self._cur_mean = f(M, A)
        self._stats = f(S['COUNT'])
        self._hyper = torch.zeros(2, dtype=torch.float64, device=dev)
        self._stop = torch.zeros(1, dtype=torch.int32, device=dev)
        L = _lib.lib()
        self._loss_ws = torch.zeros(L.sb200_ppo_loss_workspace_bytes(M, A), dtype=torch.uint8, device=dev)
        self._loss_ws_v = torch.zeros_like(self._loss_ws)     # the value branch runs concurrently with the policy branch
        self._side_stream = None
        self._rfilter_stats = torch.tensor([1e-5, 0.0, 0.0], dtype=torch.float32, device=dev) \
            if self.use_r_filter else None
        self._pin = {}
        self._gae_ws = torch.zeros(int(L.sb200_gae_workspace_bytes(B, n, n)), dtype=torch.uint8, device=dev)
        self.use_cuda_graph = ops.graphs_enabled()
        # policy || value epochs as concurrent graph branches -- not in pixel mode, where both optimisers update the SHARED stem
        self.parallel_branches = os.environ.get("SB200_PPO_FORK", "1") != "0" and not self.pixel and not self.rnn
        # tensor pipe || FMA pipe critic pass: measured SLOWER (701-757 us) than the 2-CTA/SM tensor-core tiles alone
        # (631 us) -- both kernels are issue-bound, they do not add up -- so it stays an experiment
        self.dual_critic = os.environ.get("SB200_DUAL_CRITIC", "0") == "1"
        self._graph = ops.GraphRunner()
        self._graph_head = ops.GraphRunner()
        self.before_epochs_hook = None                    # see _optimize
        self._tc5 = ops.Tc5Forward(self.model.critic)     # critic pass on tcgen05 / TMEM when the shape qualifies
        self.tc5_min_rows = int(os.environ.get('SB200_TC5_MIN_ROWS', '4096'))
        self.dp = None
        self.dp_v = None
        # all epochs of BOTH optimisers as ONE persistent kernel (csrc/epoch2.cu) instead of ~10 launches per epoch;
        # SB200_EPOCH_KERNEL=0 selects the launch chain (always the path of the pixel / RNN stems)
        self.use_epoch_kernel = os.environ.get('SB200_EPOCH_KERNEL', '2') != '0' and not self.pixel and not self.rnn
        self._ek = None
        self.epoch_kernel_gen = 2 if self.use_epoch_kernel else 0
        self.epoch_history = []
        self._sync_hyper()
        self.last_n_policy_epochs = 0
        self.profile_events = False
        self._prof = {}
        self.optimizer_steps_profiled = 0

    # ------------------------------------------------------------------------------------------------
    def _sync_hyper(self):
        self._hyper.copy_(torch.tensor([getattr(self, 'clip_epsilon', 0.0), getattr(self, 'beta', 0.0)],
                                       dtype=torch.float64))

    def _h2d(self, name, arr, dst):
        """numpy -> pinned staging -> device buffer (non-blocking); CUDA tensors are copied device-side."""
        if isinstance(arr, torch.Tensor):
            dst.copy_(arr.reshape(dst.shape), non_blocking=True)
            return 0 if arr.is_cuda else dst.numel() * 4
        a = np.asarray(arr)
        if name not in self._pin:
            self._pin[name] = torch.empty(dst.shape, dtype=torch.float32, pin_memory=True)
        self._pin[name].numpy()[...] = a.reshape(tuple(dst.shape))      # float64 -> float32 like torch.tensor(..)
        dst.copy_(self._pin[name], non_blocking=True)
        return dst.numel() * 4

    def _low_dim(self, obs):
        if isinstance(obs, dict):
            # the reference concatenates in obs_spec order (ppo_net.py:168-178), not in the batch dict's order
            keys = [k for k in self.obs_spec['low_dim'] if k in obs['low_dim']] if 'low_dim' in self.obs_spec \
                else list(obs['low_dim'])
            xs = [obs['low_dim'][k] for k in keys]
            if len(xs) == 1:
                return xs[0]
            return torch.cat(xs, -1) if isinstance(xs[0], torch.Tensor) else np.concatenate(xs, -1)
        return obs

    @staticmethod
    def _dev_ok(t, shape):
        return isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() \
            and tuple(t.shape) == tuple(shape)

    def _preprocess_batch_ppo(self, batch):
        """ppo.py:420-484: everything becomes fp32 on the device.  The learner's working layout is
        obs_full [B, n+1, D] (row n = obs_next), i.e. the reference's cat([obs, obs_next], 1) (ppo.py:380)
        done once at ingest.  A device batch from the HBM replay (which already stores windows that way) is
        used in place -- zero copies; a host batch goes through pinned staging.  Reward scaling happens inside
        the GAE / reward-filter kernel."""
        get = (lambda k: batch[k]) if isinstance(batch, dict) else (lambda k: getattr(batch, k))
        B, n, A, D = self.batch_size, self.n_step, self.action_dim, self.low_dim
        pinfo = get('persistent_infos')
        if pinfo is None:
            raise ValueError('PPO needs the behaviour policy in persistent_infos (ppo_agent.py:149)')
        full = batch.get('obs_full') if isinstance(batch, dict) else None
        own = self._own
        if self._dev_ok(full, (B, n + 1, D)) and self._dev_ok(get('actions'), (B, n, A)) and \
                self._dev_ok(pinfo[-1], (B, n, 2 * A)) and self._dev_ok(get('rewards'), (B, n)) and \
                self._dev_ok(get('dones'), (B, n)):
            # device batch (HBM replay).  When the replay gathered straight into our buffers (replay_out_buffers)
            # there is nothing to do; foreign device tensors are copied device-to-device so that the captured
            # CUDA graph always reads the same addresses.
            for src, dst in ((full, own['obs_full']), (get('actions'), own['actions']), (pinfo[-1], own['pds']),
                             (get('rewards'), own['rewards']), (get('dones'), own['dones'])):
                if src.data_ptr() != dst.data_ptr():
                    dst.copy_(src, non_blocking=True)
            self.last_h2d_bytes = 0
            return batch
        self._obs_full, self._actions, self._pds = own['obs_full'], own['actions'], own['pds']
        self._rewards, self._dones = own['rewards'], own['dones']
        nbytes = 0
        if isinstance(full, torch.Tensor) and not full.is_cuda and tuple(full.shape) == (B, n + 1, D):
            # host batch already in the working layout (ideally pinned): one DMA, no staging copy
            own['obs_full'].copy_(full, non_blocking=True)
            nbytes += own['obs_full'].numel() * 4
            obs = None
        elif self.mixed:
            obs = None
            nbytes += self._stage_mixed(get('obs'), get('obs_next'))
        elif self.pixel:
            obs = None
            fo, fn = get('obs')['pixel']['camera0'], get('obs_next')['pixel']['camera0']
            u8 = own['obs_full'].view(torch.uint8).view(B, n + 1, -1)
            if isinstance(fo, torch.Tensor):
                u8[:, :n].copy_(fo.reshape(B, n, -1), non_blocking=True)
                u8[:, n:].copy_(fn.reshape(B, 1, -1), non_blocking=True)
            else:
                if 'frames' not in self._pin:
                    self._pin['frames'] = torch.empty(B, n + 1, u8.shape[-1], dtype=torch.uint8, pin_memory=True)
                pf = self._pin['frames'].numpy()
                pf[:, :n] = np.asarray(fo, dtype=np.uint8).reshape(B, n, -1)
                pf[:, n:] = np.asarray(fn, dtype=np.uint8).reshape(B, 1, -1)
                u8.copy_(self._pin['frames'], non_blocking=True)
                nbytes += u8.numel()
        else:
            obs, obs_next = self._low_dim(get('obs')), self._low_dim(get('obs_next'))
        od = self.obs_dim
        if obs is None:
            pass
        elif isinstance(obs, torch.Tensor):
            own['obs_full'][:, :n, :od].copy_(obs.reshape(B, n, od), non_blocking=True)
            own['obs_full'][:, n:, :od].copy_(obs_next.reshape(B, 1, od), non_blocking=True)
            if self.rnn:                                          # onetime_infos = [h0, c0] of the window's first step
                hc = get('onetime_infos')
                Hh = self.model.rnn_stem.H
                own['obs_full'][:, 0, od:od + Hh].copy_(torch.as_tensor(hc[0]).reshape(B, Hh), non_blocking=True)
                own['obs_full'][:, 0, od + Hh:od + 2 * Hh].copy_(torch.as_tensor(hc[1]).reshape(B, Hh), non_blocking=True)
        else:
            if 'obs_full' not in self._pin:
                self._pin['obs_full'] = torch.zeros(B, n + 1, D, dtype=torch.float32).pin_memory()
            pf = self._pin['obs_full'].numpy()
            pf[:, :n, :od] = np.asarray(obs).reshape(B, n, od)
            pf[:, n:, :od] = np.asarray(obs_next).reshape(B, 1, od)
            if self.rnn:
                hc = get('onetime_infos')
                Hh = self.model.rnn_stem.H
                pf[:, 0, od:od + Hh] = np.asarray(hc[0], dtype=np.float32).reshape(B, Hh)
                pf[:, 0, od + Hh:od + 2 * Hh] = np.asarray(hc[1], dtype=np.float32).reshape(B, Hh)
            own['obs_full'].copy_(self._pin['obs_full'], non_blocking=True)
            nbytes += own['obs_full'].numel() * 4
        nbytes += self._h2d('actions', get('actions'), own['actions'])
        nbytes += self._h2d('rewards', get('rewards'), own['rewards'])
        nbytes += self._h2d('dones', get('dones'), own['dones'])
        nbytes += self._h2d('pds', pinfo[-1], own['pds'])
        self.last_h2d_bytes = nbytes
        return batch

    def _stage_mixed(self, obs, obs_next):
        """Mixed observation dicts (frames + low-dim keys, host or device) -> the record rows of obs_full.  Returns the bytes
        sent host-to-device."""
        B, n, lay = self.batch_size, self.n_step, self.obs_layout
        full = self._own['obs_full']
        if isinstance(obs['pixel']['camera0'], torch.Tensor):
            for src, dst in ((obs, U.mixed_obs_views(full[:, :n], lay)), (obs_next, U.mixed_obs_views(full[:, n:], lay))):
                d = dst['pixel']['camera0']
                d.copy_(src['pixel']['camera0'].reshape(d.shape), non_blocking=True)
                for k, _, _ in lay['keys']:
                    dst['low_dim'][k].copy_(src['low_dim'][k].reshape(dst['low_dim'][k].shape), non_blocking=True)
            return 0
        if 'obs_full' not in self._pin:
            self._pin['obs_full'] = torch.zeros(tuple(full.shape), dtype=torch.float32).pin_memory()
        pf = self._pin['obs_full'].numpy()
        pf[:, :n] = U.pack_obs_rows(obs, lay).reshape(B, n, -1)
        pf[:, n:] = U.pack_obs_rows(obs_next, lay).reshape(B, 1, -1)
        full.copy_(self._pin['obs_full'], non_blocking=True)
        return full.numel() * 4

    def _low_dim_cols(self):
        """Mixed mode: the low-dim columns of the record rows (a view starting at the first one; callers pass rows / ldx)."""
        return self._obs_full.view(-1)[self.obs_layout['low_dim_off']:]

    def _mixed_stem(self, trainer=None, ref=False):
        """Mixed mode: CNN features of the step-0 frame of every window, read in place from obs_full."""
        rb = 4 * (self.n_step + 1) * self.low_dim
        if trainer is not None:
            return trainer.forward(self._obs_full, row_bytes=rb)
        return self.ref_target_model.cnn_stem.forward(self._obs_full, self._ref_stem_bufs, rows=self.batch_size, row_bytes=rb)

    # ------------------------------------------------------------------------------------------------
    def _gae_and_return(self):
        """ppo.py:355-418 (MLP branch): critic over all B*(n+1) rows without materialising the cat, then GAE."""
        B, n = self.batch_size, self.n_step
        m = self.model
        ev = self._prof_begin()
        rows = B * (n + 1)
        if self.rnn:
            # the critic over the whole [B, n+1] sequence through the LSTM from the window's initial cells (ppo.py:376-387),
            # then the horizon-windowed GAE over eff_len positions (ppo.py:389-406)
            self._rnn_prepare()
            h0, c0, ld = self._cells()
            h_all = m.rnn_stem.forward(self._xf_all, h0, c0, ld, B, n + 1, self._rnn_all)
            ops.mlp_forward(m.critic, h_all, out=self._values)
        elif self.mixed:
            # all B*(n+1) frames through the shared stem in place, then the critic head on (low-dim | features)
            if self._stem_all is None:
                self._stem_all = m.cnn_stem.buffers(rows)
            D = self.low_dim
            feat = m.cnn_stem.forward(self._obs_full, self._stem_all, rows=rows, row_bytes=4 * D)
            ops.mlp_forward(m.critic, self._low_dim_cols(), zf_stats=m.z_stats, zf_eps=m.z_eps, aux=feat, rows=rows, ldx=D,
                            out=self._values)
        elif self.pixel:
            # all B*(n+1) frames through the shared stem, then the critic head on the features (ppo.py:376-387, 5-D obs)
            stem = m.cnn_stem
            if self._stem_all is None:
                self._stem_all = stem.buffers(rows)
            frames = self._obs_full.view(torch.uint8).view(rows, *stem_shape(stem))
            feat = stem.forward(frames, self._stem_all)
            if rows >= self.tc5_min_rows and self._tc5.supported(rows):
                self._tc5(feat, self._values.view(rows, 1))
            else:
                ops.mlp_forward(m.critic, feat, out=self._values)
        elif rows >= self.tc5_min_rows and self._tc5.supported(rows):
            # Blackwell-native path: tcgen05.mma tiles, accumulators in TMEM, weights streamed by the TMA engine
            self._tc5(self._obs_full.view(rows, -1), self._values.view(rows, 1), zf_stats=m.z_stats, zf_eps=m.z_eps)
        elif self.dual_critic and rows >= 32768:
            ops.mlp_forward_dual(m.critic, self._obs_full.view(rows, -1), zf_stats=m.z_stats, zf_eps=m.z_eps,
                                 out=self._values.view(rows, 1))
        else:
            ops.mlp_forward(m.critic, self._obs_full.view(rows, -1), zf_stats=m.z_stats, zf_eps=m.z_eps,
                            out=self._values)
        self._prof_end('critic_pass', ev)
        rewards, scale = self._rewards, self.reward_scale
        if self.use_r_filter:
            check(_lib.lib().sb200_reward_filter_f32(_ptr(self._rewards), B * n, float(self.reward_scale), 1e-5,
                                                     _ptr(self._rfilter_stats), _ptr(self._rewards_f), ops._stream()),
                  'sb200_reward_filter_f32')
            rewards, scale = self._rewards_f, 1.0
        ev = self._prof_begin()
        local_norm = self.norm_adv and self.dp is None
        ops.gae_window(rewards, self._values.view(B, n + 1), self._dones, self.gamma, self.lam, norm_adv=local_norm,
                       horizon=self.horizon if self.rnn else None, reward_scale=scale, adv=self._adv, ret=self._ret,
                       ws=self._gae_ws)
        if self.norm_adv and self.dp is not None:                 # statistics of the GLOBAL batch (ppo.py:413-416)
            L = _lib.lib()
            check(L.sb200_moments_f32(_ptr(self._adv), B, _ptr(self._moments), ops._stream()), 'sb200_moments_f32')
            self.dp.sum_(self._moments)
            check(L.sb200_normalize_f32(_ptr(self._adv), B, _ptr(self._moments), 1e-4, ops._stream()),
                  'sb200_normalize_f32')
        self._prof_end('gae', ev)
        return self._adv, self._ret

    # -- RNN mode helpers ---------------------------------------------------------------------------------
    def _cells(self):
        """(h0, c0, ld): the LSTM cells at the first step of every window; they ride in row 0 of the observation records
        (the reference ships them as onetime_infos, ppo_agent.py:133-137, ppo.py:507-510)."""
        od, Hh = self.obs_dim, self.model.rnn_stem.H
        return self._obs_full[:, 0, od:od + Hh], self._obs_full[:, 0, od + Hh:od + 2 * Hh], self._obs_full.stride(0)

    def _rnn_prepare(self):
        """Once per learn(): contiguous, z-filtered sequence rows -- all n+1 steps for the critic pass, the first eff_len
        for the updates (through the learner's AND the reference model's filter, ppo.py:507-539) -- and the step slices of
        actions / behaviour policy the updates iterate on."""
        from ..model.lstm_stem import rows_zfilter
        B, n, A, E, od, Dp = self.batch_size, self.n_step, self.action_dim, self.eff_len, self.obs_dim, self.low_dim
        m, ref = self.model, self.ref_target_model
        o = self._obs_full
        rows_zfilter(o, Dp, (n + 1) * Dp, B, n + 1, od, m.z_stats, m.z_eps, self._xf_all)
        rows_zfilter(o, Dp, (n + 1) * Dp, B, E, od, m.z_stats, m.z_eps, self._xf_eff)
        rows_zfilter(o, Dp, (n + 1) * Dp, B, E, od, ref.z_stats, ref.z_eps, self._xf_ref)
        rows_zfilter(o, Dp, (n + 1) * Dp, B, E, od, None, 0.0, self._xraw_eff)
        rows_zfilter(self._actions, A, n * A, B, E, A, None, 0.0, self._act_it)
        rows_zfilter(self._pds, 2 * A, n * 2 * A, B, E, 2 * A, None, 0.0, self._pd_it)

    # -- live kernel timing for bench.py's roofline (CUDA events on the launching stream) ---------------
    def _prof_begin(self):
        if not self.profile_events:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def _prof_end(self, name, e0):
        if e0 is None:
            return
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        self._prof.setdefault(name, []).append((e0, e1))

    def pop_profile(self, name):
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in self._prof.pop(name, [])]

    def replay_out_buffers(self):
        """Buffers the HBM replay gathers a sampled batch into (zero extra copies, stable addresses)."""
        o = self._own
        return dict(obs_full=o['obs_full'], actions=o['actions'], pd=o['pds'], rewards=o['rewards'], dones=o['dones'])

    def _policy_epoch(self, stop=None, fresh=True):
        """One policy epoch (ppo.py:523-556).  The post-step forward that measures KL(ref || new) runs on the same
        inputs and parameters as the NEXT epoch's training forward, so it is done once, with saved activations:
        ``fresh=False`` reuses it."""
        L = _lib.lib()
        B, n, A, D = self.batch_size, self.n_step, self.action_dim, self.low_dim
        m, tr, st = self.model, self.actor_optim, ops._stream()
        M = self._rows
        acts, lda, pds, ldp = (self._act_it, A, self._pd_it, 2 * A) if self.rnn else (self._actions, n * A, self._pds, n * 2 * A)
        if self.rnn:
            mean = tr.forward(self.actor_rnn.forward(self._xf_eff, *self._cells())) if fresh else tr.out
        elif self.mixed:
            mean = tr.forward(self._low_dim_cols(), zf_stats=m.z_stats, zf_eps=m.z_eps, aux=self._mixed_stem(self.actor_stem),
                              rows=B, ldx=(n + 1) * D) if fresh else tr.out
        elif self.pixel:
            mean = tr.forward(self.actor_stem.forward(self._frames0)) if fresh else tr.out
        else:
            mean = tr.forward(self._obs_full, zf_stats=m.z_stats, zf_eps=m.z_eps, rows=B, ldx=(n + 1) * D) if fresh \
                else tr.out
        mode = 0 if self.ppo_mode == 'clip' else 1
        if mode == 1:
            self._kl(mean, S['KL_PRE'], 0.0, stop)
        dlog_var = tr.slabs[0, m.actor.extra_off:m.actor.extra_off + A]
        check(L.sb200_ppo_policy_loss_f32(mode, _ptr(mean), mean.stride(0), _ptr(m.log_var), _ptr(acts), lda,
                                          _ptr(self._adv), _ptr(pds), ldp, _ptr(self._ref_pd), 2 * A, M, A,
                                          _ptr(self._hyper), float(self.eta), float(self.kl_target), _ptr(tr.d[-1]),
                                          tr.d[-1].stride(0), _ptr(dlog_var), _ptr(self._stats), _ptr(self._loss_ws),
                                          _ptr(stop), st), 'sb200_ppo_policy_loss_f32')
        tr.backward()
        if self.rnn:
            from ..model.cnn_stem import joint_step
            self.actor_rnn.backward(tr.dx0)
            joint_step(tr, self.actor_rnn, self._g_actor, norm_out=self._stats[S['GN_ACTOR']:S['GN_ACTOR'] + 1], stop_flag=stop)
            self._cur_mean = tr.forward(self.actor_rnn.forward(self._xf_eff, *self._cells()))
        elif self.mixed:
            from ..model.cnn_stem import joint_step
            self.actor_stem.backward(tr.dx0)
            joint_step(tr, self.actor_stem, self._g_actor, norm_out=self._stats[S['GN_ACTOR']:S['GN_ACTOR'] + 1], stop_flag=stop)
            self._cur_mean = tr.forward(self._low_dim_cols(), zf_stats=m.z_stats, zf_eps=m.z_eps,
                                        aux=self._mixed_stem(self.actor_stem), rows=B, ldx=(n + 1) * D)
        elif self.pixel:
            from ..model.cnn_stem import joint_step
            self.actor_stem.backward(tr.dx0)
            joint_step(tr, self.actor_stem, self._g_actor, norm_out=self._stats[S['GN_ACTOR']:S['GN_ACTOR'] + 1], stop_flag=stop)
            self._cur_mean = tr.forward(self.actor_stem.forward(self._frames0))
        else:
            tr.step(norm_out=self._stats[S['GN_ACTOR']:S['GN_ACTOR'] + 1], stop_flag=stop)
            # post-step KL(ref || current) (ppo.py:553-556)
            self._cur_mean = tr.forward(self._obs_full, zf_stats=m.z_stats, zf_eps=m.z_eps, rows=B, ldx=(n + 1) * D)
        self._kl(self._cur_mean, S['KL_POST'], 4.0 * self.kl_target, self._stop)

    def _kl(self, mean, slot, threshold, stop):
        """mean KL(ref || (mean, exp(log_var))) -> stats[slot]; raises the stop flag above `threshold`.  With a
        data-parallel learner the scalar is averaged over ranks between the two halves."""
        L = _lib.lib()
        B, A, m, st = self._rows, self.action_dim, self.model, ops._stream()
        dp = self.dp
        check(L.sb200_ppo_kl_f32(_ptr(self._ref_pd), 2 * A, _ptr(mean), mean.stride(0), _ptr(m.log_var), B, A,
                                 _ptr(self._stats), slot, float(threshold), _ptr(stop), 0 if dp is None else 1,
                                 _ptr(self._loss_ws), st), 'sb200_ppo_kl_f32')
        if dp is not None:
            dp.mean_(self._kl_scalar)
            check(L.sb200_ppo_kl_apply(_ptr(self._loss_ws), _ptr(self._stats), slot, float(threshold), _ptr(stop), st),
                  'sb200_ppo_kl_apply')

    def enable_data_parallel(self, group=None):
        """Shard the learner's batch over the ranks of `group` (SURVEY §8e): this rank keeps its own actors / replay
        shard / B local windows; gradients, advantage moments, the KL scalar, z-filter sums and statistics are
        all-reduced.  Parameters start from rank 0's initialisation."""
        from ..parallel import LearnerDP
        if self.use_r_filter:
            raise NotImplementedError('reward filter + data parallel')
        if self.rnn:
            raise NotImplementedError('RNN mode + data parallel')
        if self.mixed:
            raise NotImplementedError('mixed pixel + low-dim observations + data parallel')
        stem_n = self.model.cnn_stem.size if self.pixel else 0
        peer_floats = max(self.model.actor.size, self.model.critic.size) + stem_n + 64
        self.dp = LearnerDP(group, peer_floats=peer_floats)
        # the value branch gets its OWN communicator: with the policy || value fork both branches issue collectives
        # concurrently, and two streams must never interleave on one communicator
        import torch.distributed as dist
        self.dp_v = LearnerDP(dist.new_group(ranks=list(range(self.dp.world))), peer_floats=peer_floats) \
            if self.parallel_branches else self.dp
        self.actor_optim.dp = self.dp
        self.critic_optim.dp = self.dp_v
        for mdl in (self.model, self.ref_target_model):
            self.dp.broadcast_(mdl.actor.params)
            self.dp.broadcast_(mdl.critic.params)
            if mdl.z_stats is not None:
                self.dp.broadcast_(mdl.z_stats)
        off = _lib.lib().sb200_ppo_loss_kl_offset()
        self._kl_scalar = self._loss_ws[off:off + 8].view(torch.float64)
        self._moments = torch.zeros(3, dtype=torch.float64, device=self.device)
        self._z_delta = torch.zeros_like(self.model.z_stats) if self.model.z_stats is not None else None
        self._graph = ops.GraphRunner()
        self._graph_head = ops.GraphRunner()
        # One CUDA graph for the whole data-parallel learn(), NCCL collectives included (SB200_DP_GRAPH=0: the same
        # launches eagerly).  Capture stays on ONE stream (no dW side stream) and every collective shape is issued
        # once eagerly first: NCCL sets up its channels lazily, which must not happen under capture.
        # (validated on 2 GPUs: same parameters / statistics as the oracle on the global batch; learn() 5.2 -> 3.7 ms.)
        # NOTE: a process that captured NCCL work must leave with os._exit() -- ProcessGroupNCCL's teardown hangs
        # (bench.py, tests/dp_check.py).  The policy || value fork is kept: the value branch reduces on its own
        # communicator (dp_v).  The dW side stream carries no collective.
        self.dp_graph = os.environ.get('SB200_DP_GRAPH', '1') != '0'
        for t in (self.actor_optim.grad, self.critic_optim.grad, self._kl_scalar, self._moments, self._z_delta,
                  self._stats):
            if t is not None:
                self.dp.sum_(torch.zeros_like(t))
        if self.dp_v is not self.dp:
            self.dp_v.sum_(torch.zeros_like(self.critic_optim.grad))
        torch.cuda.synchronize()
        return self

    def _value_epoch(self):
        L = _lib.lib()
        B, n, D = self.batch_size, self.n_step, self.low_dim
        m, tr, st = self.model, self.critic_optim, ops._stream()
        if self.rnn:
            v = tr.forward(self.critic_rnn.forward(self._xf_eff, *self._cells()))
        elif self.mixed:
            v = tr.forward(self._low_dim_cols(), zf_stats=m.z_stats, zf_eps=m.z_eps, aux=self._mixed_stem(self.critic_stem),
                           rows=B, ldx=(n + 1) * D)
        elif self.pixel:
            v = tr.forward(self.critic_stem.forward(self._frames0))
        else:
            v = tr.forward(self._obs_full, zf_stats=m.z_stats, zf_eps=m.z_eps, rows=B, ldx=(n + 1) * D)
        check(L.sb200_value_loss_f32(_ptr(v), v.stride(0), _ptr(self._ret), self._rows, _ptr(tr.d[-1]), tr.d[-1].stride(0),
                                     _ptr(self._stats), _ptr(self._loss_ws_v), st), 'sb200_value_loss_f32')
        tr.backward()
        if self.rnn:
            from ..model.cnn_stem import joint_step
            self.critic_rnn.backward(tr.dx0)
            joint_step(tr, self.critic_rnn, self._g_critic, norm_out=self._stats[S['GN_CRITIC']:S['GN_CRITIC'] + 1])
        elif self.pixel:                                          # pixel and mixed: the stem takes the features' gradient
            from ..model.cnn_stem import joint_step
            self.critic_stem.backward(tr.dx0)
            joint_step(tr, self.critic_stem, self._g_critic, norm_out=self._stats[S['GN_CRITIC']:S['GN_CRITIC'] + 1])
        else:
            tr.step(norm_out=self._stats[S['GN_CRITIC']:S['GN_CRITIC'] + 1])

    def _optimize_head(self):
        B, n, A, D = self.batch_size, self.n_step, self.action_dim, self.low_dim
        ref = self.ref_target_model
        self._gae_and_return()
        if self.rnn:
            h_ref = ref.rnn_stem.forward(self._xf_ref, *self._cells(), B, self.eff_len, self._rnn_ref)
            ops.mlp_forward(ref.actor, h_ref, out=self._ref_mean)
        elif self.mixed:
            ops.mlp_forward(ref.actor, self._low_dim_cols(), zf_stats=ref.z_stats, zf_eps=ref.z_eps, aux=self._mixed_stem(ref=True),
                            rows=B, ldx=(n + 1) * D, out=self._ref_mean)
        elif self.pixel:
            # step-0 frames of every window, contiguous (ppo.py:527-537), then the reference policy on them
            fr = self._obs_full.view(torch.uint8).view(B, n + 1, -1)
            self._frames0.view(B, -1).copy_(fr[:, 0])
            ops.mlp_forward(ref.actor, ref.cnn_stem.forward(self._frames0, self._ref_stem_bufs), out=self._ref_mean)
        else:
            ops.mlp_forward(ref.actor, self._obs_full, zf_stats=ref.z_stats, zf_eps=ref.z_eps, rows=B, ldx=(n + 1) * D,
                            out=self._ref_mean)
        ops.make_pd(self._ref_mean, ref.log_var, self._rows, A, self._ref_pd)
        self._stats.zero_()
        self._stop.zero_()

    def _optimize_tail(self, value_done=False):
        L = _lib.lib()
        B, n, A, D = self.batch_size, self.n_step, self.action_dim, self.low_dim
        m, st = self.model, ops._stream()
        if not value_done:
            for _ in range(self.epoch_baseline):
                self._value_epoch()
        acts, lda, pds, ldp = (self._act_it, A, self._pd_it, 2 * A) if self.rnn else (self._actions, n * A, self._pds, n * 2 * A)
        check(L.sb200_ppo_final_stats_f32(_ptr(self._cur_mean), self._cur_mean.stride(0), _ptr(m.log_var),
                                          _ptr(acts), lda, _ptr(pds), ldp, _ptr(self._ref_pd), 2 * A, self._rows, A,
                                          _ptr(self._stats), _ptr(self._loss_ws), st), 'sb200_ppo_final_stats_f32')
        if self.use_z_filter:
            # the rows the updates trained on (step 0 of every window; the first eff_len steps in RNN mode), AFTER the
            # updates (ppo.py:578)
            if self.rnn:
                ops.zfilter_update(self._xraw_eff, self._rows, self.obs_dim, self._xraw_eff.stride(0), m.z_stats)
            elif self.mixed:
                ops.zfilter_update(self._low_dim_cols(), B, self.obs_dim, (n + 1) * D, m.z_stats)
            elif self.dp is None:
                ops.zfilter_update(self._obs_full, B, D, (n + 1) * D, m.z_stats)
            else:
                self._z_delta.zero_()
                ops.zfilter_update(self._obs_full, B, D, (n + 1) * D, self._z_delta)
                self.dp.sum_(self._z_delta)
                check(L.sb200_add_f32(_ptr(m.z_stats), _ptr(self._z_delta), 2 * D + 1, st), 'sb200_add_f32')
        if self.dp is not None:
            self.dp.mean_(self._stats)                            # every slot is a batch mean (or rank-invariant)

    def _epoch_kernels(self):
        """(policy, value) persistent-kernel bindings over the current batch buffers, or None when this configuration
        takes the launch chain (pixel / RNN stems, unsupported layer shapes, NCCL-only data parallel)."""
        if not self.use_epoch_kernel:
            return None
        if self.dp is not None and (self.dp.peer is None or self.dp_v.peer is None):
            return None
        if self.model.actor.n_layers != 3 or self.model.critic.n_layers != 3:
            return None                                           # the kernel is written for input -> 2 hidden -> head
        B, n, A, D = self.batch_size, self.n_step, self.action_dim, self.low_dim
        key = (self._obs_full.data_ptr(), self._actions.data_ptr(), self._pds.data_ptr(), id(self.dp))
        if self._ek is None or self._ek[0] != key:
            m = self.model
            mode = 0 if self.ppo_mode == 'clip' else 1
            pk = ops.EpochKernel(self.actor_optim, mode, self._obs_full, (n + 1) * D, B, m.z_stats, m.z_eps, self._stats,
                                 self.epoch_policy, norm_out=self._stats[S['GN_ACTOR']:S['GN_ACTOR'] + 1], stop_flag=self._stop,
                                 actions=self._actions, lda=n * A, adv=self._adv, behave_pd=self._pds, ldb=n * 2 * A,
                                 ref_pd=self._ref_pd, ldr=2 * A, hyper=self._hyper, eta=self.eta, kl_target=self.kl_target,
                                 stop_threshold=4.0 * self.kl_target, cta_shift=0)
            vk = ops.EpochKernel(self.critic_optim, 2, self._obs_full, (n + 1) * D, B, m.z_stats, m.z_eps, self._stats,
                                 self.epoch_baseline, norm_out=self._stats[S['GN_CRITIC']:S['GN_CRITIC'] + 1],
                                 returns=self._ret)
            if self.dp is not None:
                pk.set_peer(self.dp.peer)
                vk.set_peer(self.dp_v.peer)
            # both optimisers in ONE launch; data-parallel needs two distinct channels (both exchange in the same phase)
            pair = None
            if (self.dp is None or self.dp_v is not self.dp) and ops.EpochPair.supported(pk, vk):
                pair = ops.EpochPair(pk, vk)
            self._ek = (key, pk, vk, pair)
        if self._ek[3] is None:
            return None                                           # shape the kernel rejects: launch chain
        return self._ek[1], self._ek[2], self._ek[3]

    def _optimize_device(self):
        """The whole of ppo.py:487-586 as one fixed launch sequence (CUDA-graph body).  The KL early stop
        (ppo.py:556) is a DEVICE flag: the post-step KL kernel raises it, and the loss / reduce / Adam / KL
        kernels of the remaining policy epochs turn into no-ops -- same parameters and statistics as breaking
        out of the loop, without a host round trip per epoch."""
        self._optimize_head()
        self._optimize_epochs()

    def _optimize_epochs(self):
        """Everything of _optimize_device behind the head (critic pass, GAE, reference-policy forward): the epochs and
        the closing statistics.  A separate graph when `before_epochs_hook` is set (see _optimize)."""
        # The value epochs (critic, returns) and the policy epochs (actor, advantages) share nothing but read-only
        # inputs: they run as two concurrent branches (a fork / join inside the captured graph), so the step costs
        # max(policy chain, value chain) instead of their sum.  With a data-parallel learner both branches would
        # issue collectives on one communicator, so that case stays sequential.
        fork = self.parallel_branches and not self.profile_events and \
            (self.dp is None or (self.dp_graph and self.dp_v is not self.dp))
        ek = self._epoch_kernels()
        if ek is not None:
            # one persistent kernel (all epochs of both optimisers, early stop and -- data-parallel -- the exchanges inside)
            self._cur_mean = ek[2].run()
            self._optimize_tail(value_done=True)
            return
        if fork:
            if self._side_stream is None:
                self._side_stream = torch.cuda.Stream(device=self.device)
            main, side = torch.cuda.current_stream(), self._side_stream
            side.wait_stream(main)
            with torch.cuda.stream(side):
                for _ in range(self.epoch_baseline):
                    self._value_epoch()
        for e in range(self.epoch_policy):
            self._policy_epoch(stop=self._stop, fresh=(e == 0))
        if fork:
            main.wait_stream(side)
        self._optimize_tail(value_done=fork)

    def _optimize(self):
        """ppo.py:487-586."""
        B, n, A, D = self.batch_size, self.n_step, self.action_dim, self.low_dim
        m = self.model
        if self.use_cuda_graph and not self.profile_events and (self.dp is None or self.dp_graph):
            ek = self._epoch_kernels()
            if self.before_epochs_hook is not None and ek is not None and ek[2] is not None:
                # The one-launch learner kernel wants every SM (a grid barrier needs all its CTAs resident), and so does the
                # actors' persistent rollout kernel: launched side by side each holds SMs the other one waits for
                # (measured: the rollout stretched from 1.5 to 2.5 ms).  A caller that runs actors concurrently
                # (PipelinedEngine) therefore gets two graphs with a hook in between: the head overlaps the rollout on the
                # SMs it leaves free, the hook waits for the rollout, then the epochs have the GPU to themselves.
                self._graph_head.run(self._optimize_head)
                self.before_epochs_hook()
                self._graph.run(self._optimize_epochs)
            else:
                self._graph.run(self._optimize_device)
        elif self.use_cuda_graph or (self._epoch_kernels() or (None, None, None))[2] is not None:
            self._optimize_device()                               # same sequence, eager (per-kernel event timing, ncu launch lists)
        else:
            self._optimize_head()                                 # reference-style host loop: one sync per epoch
            for e in range(self.epoch_policy):
                self._policy_epoch(fresh=(e == 0))
                if float(self._stats[S['KL_POST']].item()) > self.kl_target * 4:
                    break
            self._optimize_tail()
        s = self._stats.cpu().numpy()                             # single D2H of all statistics
        self.last_d2h_bytes = s.nbytes
        n_ep = int(round(float(s[S['EPOCHS']])))
        self.last_n_policy_epochs = n_ep
        self.epoch_history.append(n_ep + self.epoch_baseline)
        self.kl_record.append(float(s[S['KL_POST']]))
        if self.profile_events:
            self.optimizer_steps_profiled += n_ep + self.epoch_baseline
        stats = {'_surr_loss': float(s[S['SURR']]), '_entropy': float(s[S['ENTROPY']])}
        if self.ppo_mode == 'clip':
            stats['_clip_surr_loss'] = float(s[S['LOSS']])
            stats['_clip_epsilon'] = self.clip_epsilon
        else:
            stats['_kl_loss_adapt'] = float(s[S['LOSS']])
            stats['_beta'] = self.beta
        if self.clip_actor_gradient:
            stats['grad_norm_actor'] = float(s[S['GN_ACTOR']])
        stats['_pol_kl'] = float(s[S['KL_POST']])
        stats['_val_loss'] = float(s[S['VAL_LOSS']])
        stats['_val_explained_var'] = float(s[S['EXPL_VAR']])
        if self.dp is not None:
            # global-batch explained variance (ppo.py:323-331) from the rank-averaged raw moments
            mo = s[S['VAL_MOMENTS']:S['VAL_MOMENTS'] + 8].astype(np.float64)
            md, md2, mr, mr2 = (mo[0] + mo[1], mo[2] + mo[3], mo[4] + mo[5], mo[6] + mo[7])
            ng = float(self.batch_size * self.dp.world)
            var_d, var_r = (md2 - md * md) * ng / (ng - 1.0), (mr2 - mr * mr) * ng / (ng - 1.0)
            stats['_val_explained_var'] = float(1.0 - var_d / var_r)
        if self.clip_critic_gradient:
            stats['grad_norm_critic'] = float(s[S['GN_CRITIC']])
        stats['_avg_return_targ'] = float(s[S['RET_MEAN']])
        stats['_avg_log_sig'] = float(s[S['LOG_SIG']])
        stats['_avg_behave_likelihood'] = float(s[S['BEHAVE_LIK']])
        stats['_avg_is_weight'] = float(s[S['IS_WEIGHT']])
        stats['_ref_behave_diff'] = float(s[S['REF_BEHAVE']])
        stats['_lr'] = self.actor_lr_scheduler.get_lr()[0]
        if self.use_z_filter:
            z = m.z_stats.cpu().double().numpy()
            D = self.obs_dim
            zs, zq, zc = z[:D], z[D:2 * D], z[2 * D]
            stats['obs_running_mean'] = float(np.mean((zs / zc).astype(np.float32)))
            stats['obs_running_square'] = float(np.mean((zq / zc).astype(np.float32)))
            stats['obs_running_std'] = float(np.mean(np.sqrt((zq / zc) - (zs / zc) ** 2).astype(np.float32)))
        if self.use_r_filter:
            rf = self._rfilter_stats.cpu().numpy()
            stats['reward_mean'] = float(rf[1] / rf[0])
        return stats

    # ------------------------------------------------------------------------------------------------
    def learn(self, batch):
        """ppo.py:588-613."""
        self.current_iteration += 1
        self._preprocess_batch_ppo(batch)
        stats = self._optimize()
        self.periodic_checkpoint(global_steps=self.current_iteration, score=None)
        self.tensorplex.add_scalars(stats, self.global_step)
        self.exp_counter += self.batch_size
        self.global_step += 1
        return stats

    def module_dict(self):
        return {'ppo': self.model}

    def publish_parameter(self, iteration, message=''):
        """ppo.py:623-635: publish only once exp_interval experiences were consumed."""
        if self.exp_counter >= self.learner_config.parameter_publish.exp_interval:
            self._ps_publisher.publish(iteration, message=message)
            self._post_publish()

    def _post_publish(self):
        """ppo.py:637-666."""
        final_kl = np.mean(self.kl_record)
        lc = self.learner_config
        if self.ppo_mode == 'clip':
            if final_kl > self.kl_target * self.clip_adjust_threshold[1]:
                if self.clip_lower < self.clip_epsilon:
                    self.clip_epsilon = self.clip_epsilon / lc.algo.clip_consts.scale_constant
            elif final_kl < self.kl_target * self.clip_adjust_threshold[0]:
                if self.clip_upper > self.clip_epsilon:
                    self.clip_epsilon = self.clip_epsilon * lc.algo.clip_consts.scale_constant
        else:
            if final_kl > self.kl_target * self.beta_adjust_threshold[1]:
                if self.beta_upper > self.beta:
                    self.beta = self.beta * lc.algo.adapt_consts.scale_constant
            elif final_kl < self.kl_target * self.beta_adjust_threshold[0]:
                if self.beta_lower < self.beta:
                    self.beta = self.beta / lc.algo.adapt_consts.scale_constant
        self._sync_hyper()
        self.ref_target_model.update_target_params(self.model)
        self.kl_record = []
        self.exp_counter = 0
        self.actor_lr_scheduler.step()
        self.critic_lr_scheduler.step()

    def checkpoint_attributes(self):
        """ppo.py:668-678.  With ``session_config.checkpoint.learner.include_optimizer`` (an extension, off by default
        so that the files keep the reference's attribute list) the Adam state and the publish-time adaptation state are
        tracked too, which makes a restored learner continue BIT-identically."""
        attrs = ['model', 'ref_target_model', 'actor_lr_scheduler', 'critic_lr_scheduler', 'current_iteration']
        ck = self.session_config.checkpoint.learner
        if 'include_optimizer' in ck and ck.include_optimizer:
            attrs += ['actor_optim', 'critic_optim', 'adapt_state']
        return attrs

    @property
    def adapt_state(self):
        return {'clip_epsilon': getattr(self, 'clip_epsilon', None), 'beta': getattr(self, 'beta', None),
                'exp_counter': self.exp_counter, 'kl_record': list(self.kl_record), 'global_step': self.global_step,
                'rfilter': self._rfilter_stats.cpu() if self._rfilter_stats is not None else None}

    @adapt_state.setter
    def adapt_state(self, st):
        if st.get('clip_epsilon') is not None:
            self.clip_epsilon = st['clip_epsilon']
        if st.get('beta') is not None:
            self.beta = st['beta']
        self.exp_counter, self.kl_record, self.global_step = st['exp_counter'], list(st['kl_record']), st['global_step']
        if st.get('rfilter') is not None and self._rfilter_stats is not None:
            self._rfilter_stats.copy_(st['rfilter'].to(self.device))
        self._sync_hyper()

    def _prefetcher_preprocess(self, batch):
        if isinstance(batch, dict):          # the HBM replay already returns an aggregated device batch
            return batch
        return self.aggregator.aggregate(batch)
