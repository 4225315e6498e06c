"""PPO actor / critic / z-filter as flat device buffers (host-side mirror of surreal/model/ppo_net.py:94-375,
model_builders/builders.py:86-175, z_filter.py:7-107).  Every forward is one fused CUDA launch."""
import collections

import torch

from .. import ops


class DiagGauss:
    """Shape bookkeeping only; the distribution math runs inside the loss kernels (csrc/ppo_loss.cu)."""

    def __init__(self, action_dim):
        self.d = action_dim


def _default_linear_init(dims, seed_gen=None):
    """torch.nn.Linear's default initialisation (the un-vendored torchx L.Linear default is unknown,
    SURVEY §8c; parity tests always inject weights)."""
    layers = []
    for i in range(len(dims) - 1):
        lin = torch.nn.Linear(dims[i], dims[i + 1])
        layers.append((lin.weight.detach().clone(), lin.bias.detach().clone()))
    return layers


class PPOModel:
    """Same constructor keywords as the reference's PPOModel (ppo_net.py:110-118).  The LSTM stem is a
    'next' row of SURVEY §8f and raises here; the CNN stem (pixel input) is model/cnn_stem.py.  With pixel input AND
    low-dim inputs (mixed observations) the heads' layer 0 takes the low-dim columns followed by the CNN features."""

    def __init__(self, obs_spec, action_dim, model_config, use_cuda=True, init_log_sig=0, use_z_filter=False,
                 if_pixel_input=False, rnn_config=None, device=None):
        self.device = torch.device(device if device is not None else 'cuda')
        if self.device.type != 'cuda':
            raise RuntimeError('surreal_b200 has no CPU path: PPOModel needs a CUDA device')
        self.obs_spec, self.action_dim, self.model_config = obs_spec, action_dim, model_config
        self.use_z_filter, self.init_log_sig = use_z_filter, init_log_sig
        self.if_pixel_input, self.rnn_config = if_pixel_input, rnn_config
        self.cnn_stem = None
        self.rnn_stem = None
        self.if_rnn = bool(rnn_config is not None and rnn_config.if_rnn_policy)
        self.low_dim = 0
        if 'low_dim' in obs_spec:
            for key in obs_spec['low_dim']:
                self.low_dim += obs_spec['low_dim'][key][0]
        # mixed observations (a camera frame AND low-dim inputs): the heads see cat([zfilter(low_dim), cnn_features], -1)
        # (ppo_net.py:262-275); here the features are the aux input of layer 0, next to the low-dim columns
        self.mixed = bool(if_pixel_input and self.low_dim > 0)
        if if_pixel_input:
            # optional CNN stem feature extractor (ppo_net.py:136-140), shared by actor and critic
            from .cnn_stem import CNNStem
            self.cnn_stem = CNNStem(obs_spec['pixel']['camera0'], model_config.cnn_feature_dim, self.device)
        in_dim = self.low_dim + (model_config.cnn_feature_dim if if_pixel_input else 0)
        if self.if_rnn:
            # optional LSTM stem feature extractor (ppo_net.py:143-152), shared by actor and critic
            if if_pixel_input:
                raise NotImplementedError('CNN + LSTM stems together (pixel input with if_rnn_policy) are not built')
            from .lstm_stem import LSTMStem
            self.rnn_stem = LSTMStem(in_dim, rnn_config.rnn_hidden, self.device, layers=rnn_config.rnn_layer)
            in_dim = rnn_config.rnn_hidden
        D, A = in_dim, action_dim
        ah, ch = list(model_config.actor_fc_hidden_sizes), list(model_config.critic_fc_hidden_sizes)
        R, T, N = ops.ACT_RELU, ops.ACT_TANH, ops.ACT_NONE
        aux = dict(aux_layer=0, aux_dim=model_config.cnn_feature_dim) if self.mixed else {}
        Dx = self.low_dim if self.mixed else D
        self.actor = ops.FlatNet([Dx] + ah + [A], [R] * len(ah) + [T], self.device, extra=A, **aux)
        self.critic = ops.FlatNet([Dx] + ch + [1], [R] * len(ch) + [N], self.device, **aux)
        self.actor.load_layers(_default_linear_init([D] + ah + [A]), extra=torch.zeros(A) + init_log_sig)
        self.critic.load_layers(_default_linear_init([D] + ch + [1]))
        self.z_eps = 1e-5
        self.z_stats = None
        if use_z_filter:
            assert self.low_dim > 0, 'No low dimensional input, please turn off z-filter'
            self.z_stats = torch.cat([torch.zeros(self.low_dim), self.z_eps * torch.ones(self.low_dim),
                                      torch.tensor([self.z_eps])]).to(self.device)

    # -- parameters --------------------------------------------------------------------------------
    @property
    def log_var(self):
        return self.actor.extra_view()

    def update_target_params(self, net):
        """ppo_net.py:226-242: actor, critic and z-filter."""
        self.actor.params.copy_(net.actor.params)
        self.critic.params.copy_(net.critic.params)
        if self.cnn_stem is not None:
            self.cnn_stem.params.copy_(net.cnn_stem.params)
        if self.rnn_stem is not None:
            self.rnn_stem.params.copy_(net.rnn_stem.params)
        if self.use_z_filter:
            self.z_stats.copy_(net.z_stats)

    def update_target_z_filter(self, net):
        if self.use_z_filter:
            self.z_stats.copy_(net.z_stats)

    def flat_state(self):
        """The raw device buffers (kernel layout) -- what the collapsed parameter wire ships."""
        st = {'actor': self.actor.params, 'critic': self.critic.params}
        if self.cnn_stem is not None:
            st['cnn_stem'] = self.cnn_stem.params
        if self.rnn_stem is not None:
            st['rnn_stem'] = self.rnn_stem.params
        if self.use_z_filter:
            st['z_stats'] = self.z_stats
        return st

    def load_flat_state(self, st):
        self.actor.params.copy_(st['actor'])
        self.critic.params.copy_(st['critic'])
        if self.cnn_stem is not None and 'cnn_stem' in st:
            self.cnn_stem.params.copy_(st['cnn_stem'])
        if self.rnn_stem is not None and 'rnn_stem' in st:
            self.rnn_stem.params.copy_(st['rnn_stem'])
        if self.use_z_filter and 'z_stats' in st:
            self.z_stats.copy_(st['z_stats'])

    def state_dict(self):
        """Keys follow the reference module tree (actor.log_var, actor.model.*, critic.model.*, z_filter.*);
        Linear weights are exported in torch's [out, in] convention."""
        sd = collections.OrderedDict()
        if self.cnn_stem is not None:
            for k, v in self.cnn_stem.state_items():
                sd[k] = v
        if self.rnn_stem is not None:
            for k, v in self.rnn_stem.state_items():
                sd[k] = v
        sd['actor.log_var'] = self.log_var.detach().clone().view(1, -1)
        for name, net in (('actor', self.actor), ('critic', self.critic)):
            for l in range(net.n_layers):
                w, b = net.get_layer(l)
                sd['%s.model.seq.%d.weight' % (name, 2 * l)] = w
                sd['%s.model.seq.%d.bias' % (name, 2 * l)] = b
        if self.use_z_filter:
            D = self.low_dim
            sd['z_filter.running_sum'] = self.z_stats[:D].clone()
            sd['z_filter.running_sumsq'] = self.z_stats[D:2 * D].clone()
            sd['z_filter.count'] = self.z_stats[2 * D:].clone()
        return sd

    def load_state_dict(self, sd):
        g = lambda k: torch.as_tensor(sd[k], dtype=torch.float32)  # noqa: E731
        if self.cnn_stem is not None:
            self.cnn_stem.load_state(sd)
        if self.rnn_stem is not None:
            self.rnn_stem.load_torch(sd, prefix='rnn_stem.')
        self.log_var.copy_(g('actor.log_var').reshape(-1).to(self.device))
        for name, net in (('actor', self.actor), ('critic', self.critic)):
            for l in range(net.n_layers):
                net.set_layer(l, g('%s.model.seq.%d.weight' % (name, 2 * l)), g('%s.model.seq.%d.bias' % (name, 2 * l)))
        if self.use_z_filter and 'z_filter.count' in sd:
            self.z_stats.copy_(torch.cat([g('z_filter.running_sum').reshape(-1), g('z_filter.running_sumsq').reshape(-1),
                                          g('z_filter.count').reshape(-1)]).to(self.device))

    # -- forward -----------------------------------------------------------------------------------
    @staticmethod
    def _flat(obs):
        if isinstance(obs, dict):
            xs = [obs['low_dim'][k] for k in obs['low_dim']]
            return xs[0] if len(xs) == 1 else torch.cat(xs, -1)
        return obs

    def _features(self, obs):
        """Pixel mode: uint8 frames [rows, C, H, W] -> CNN features (ppo_net.py:268-273,368-375)."""
        fr = obs['pixel']['camera0'] if isinstance(obs, dict) else obs
        fr = fr.reshape(-1, *fr.shape[-3:]).contiguous()
        rows = fr.shape[0]
        if getattr(self, '_stem_bufs_rows', None) != rows:
            self._stem_bufs, self._stem_bufs_rows = self.cnn_stem.buffers(rows), rows
        return self.cnn_stem.forward(fr, self._stem_bufs)

    def _mixed_inputs(self, obs):
        """Mixed mode: (low-dim rows [rows, Dl], CNN features [rows, F]) of an observation dict."""
        x = self._flat(obs)
        return x.reshape(-1, x.shape[-1]).contiguous(), self._features(obs)

    def forward_actor(self, obs, cells=None, out_pd=None):
        """-> [rows, 2A] = cat(mean, std) (builders.py:114-132)."""
        if self.mixed:
            x2, feat = self._mixed_inputs(obs)
            mean = ops.mlp_forward(self.actor, x2, zf_stats=self.z_stats, zf_eps=self.z_eps, aux=feat)
            B, A = mean.shape[0], self.action_dim
            pd = out_pd if out_pd is not None else torch.empty(B, 2 * A, dtype=torch.float32, device=self.device)
            ops.make_pd(mean, self.log_var, B, A, pd)
            return pd
        if self.cnn_stem is not None:
            x2 = self._features(obs)
            mean = ops.mlp_forward(self.actor, x2)
            B, A = mean.shape[0], self.action_dim
            pd = out_pd if out_pd is not None else torch.empty(B, 2 * A, dtype=torch.float32, device=self.device)
            ops.make_pd(mean, self.log_var, B, A, pd)
            return pd
        x = self._flat(obs)
        x2 = x.reshape(-1, x.shape[-1])
        mean = ops.mlp_forward(self.actor, x2, zf_stats=self.z_stats, zf_eps=self.z_eps)
        B, A = mean.shape[0], self.action_dim
        pd = out_pd if out_pd is not None else torch.empty(B, 2 * A, dtype=torch.float32, device=self.device)
        ops.make_pd(mean, self.log_var, B, A, pd)
        return pd

    def forward_critic(self, obs, cells=None):
        if self.mixed:
            x2, feat = self._mixed_inputs(obs)
            return ops.mlp_forward(self.critic, x2, zf_stats=self.z_stats, zf_eps=self.z_eps, aux=feat)
        if self.cnn_stem is not None:
            return ops.mlp_forward(self.critic, self._features(obs))
        x = self._flat(obs)
        x2 = x.reshape(-1, x.shape[-1])
        return ops.mlp_forward(self.critic, x2, zf_stats=self.z_stats, zf_eps=self.z_eps)

    def z_update(self, obs):
        if not self.use_z_filter:
            raise ValueError('Z_update called when network is set to not use z_filter')
        x = self._flat(obs)
        x2 = x.reshape(-1, x.shape[-1])
        ops.zfilter_update(x2, x2.shape[0], self.low_dim, x2.stride(0), self.z_stats)
