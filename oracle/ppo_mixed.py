"""PPO learner restatement, MIXED observations: a camera frame and low-dim inputs (reference: surreal/model/ppo_net.py:
130-166,262-282; the default PPO env config asks for this, ppo_configs.py:111-114).  The frame goes through the shared CNN stem
of the pixel oracle, the low-dim inputs (concatenated in obs_spec order) through the z-filter, and actor and critic see
cat([zfilter(low_dim), cnn_features], -1).

An observation is carried as ONE float row [frame pixels (0..255) | low-dim floats], so that the parent classes' slicing
(obs[:, 0, :], the cat of obs and obs_next) works unchanged; the z-filter only ever sees the low-dim columns.

TEST INFRASTRUCTURE (like the rest of oracle/): stock torch on the CPU, the same call sequence as the reference.
"""
import numpy as np
import torch

from . import nets
from .ppo_pixel import OraclePPOLearnerPixel


class _LowDimZFilter:
    """A ZFilter applied to the trailing low-dim columns of a mixed observation row."""

    def __init__(self, zf, start):
        self.zf, self.start = zf, start

    def clone(self):
        return _LowDimZFilter(self.zf.clone(), self.start)

    def forward(self, x):
        return self.zf.forward(x[..., self.start:])

    def update(self, x):
        self.zf.update(x[..., self.start:])

    def running_mean(self):
        return self.zf.running_mean()

    def running_square(self):
        return self.zf.running_square()

    def running_std(self):
        return self.zf.running_std()


class OraclePPOLearnerMixed(OraclePPOLearnerPixel):
    def __init__(self, actor_layers, log_var, critic_layers, zfilter, conv_layers, strides, fc_layer, frame_shape,
                 action_dim, n_step, batch_size, **cfg):
        """As OraclePPOLearnerPixel, plus ``zfilter`` (oracle.filters.ZFilter over the low-dim inputs, or None) and
        ``frame_shape`` (C, H, W).  Layer 0 of actor and critic takes Dl + F inputs: low-dim first, then the features."""
        super().__init__(actor_layers, log_var, critic_layers, conv_layers, strides, fc_layer, action_dim, n_step, batch_size,
                         **cfg)
        self.frame_shape = tuple(int(v) for v in frame_shape)
        self.P = int(np.prod(self.frame_shape))
        self.zf = _LowDimZFilter(zfilter.clone(), self.P) if zfilter is not None else None
        self.ref_zf = self.zf.clone() if self.zf is not None else None

    def flat(self, obs):
        """{'pixel': {'camera0': [..., C, H, W]}, 'low_dim': {key: [..., w]}} -> float32 rows [..., P + Dl] (numpy)."""
        fr = np.asarray(obs['pixel']['camera0'])
        lead = fr.shape[:fr.ndim - 3]
        parts = [fr.reshape(lead + (self.P,)).astype(np.float32)]
        parts += [np.asarray(v, dtype=np.float32).reshape(lead + (-1,)) for v in obs['low_dim'].values()]
        return np.concatenate(parts, -1)

    def preprocess(self, batch):
        return super().preprocess(dict(batch, obs=self.flat(batch['obs']), obs_next=self.flat(batch['obs_next'])))

    def _inputs(self, obs, ref=False):
        zf = self.ref_zf if ref else self.zf
        low = obs[..., self.P:]
        x = zf.forward(obs) if zf is not None else low                      # ppo_net.py:262-266
        feat = self.stem(obs[..., :self.P].reshape(-1, *self.frame_shape), ref)   # ppo_net.py:268-273
        return torch.cat([x.reshape(-1, x.shape[-1]), feat], -1)            # ppo_net.py:275

    def forward_actor(self, obs, ref=False):
        h = self._inputs(obs, ref)
        if ref:
            return nets.ppo_actor(h, self.ref_actor, self.ref_log_var)
        return nets.ppo_actor(h, self.actor, self.log_var)

    def forward_critic(self, obs):
        return nets.ppo_critic(self._inputs(obs), self.critic)
