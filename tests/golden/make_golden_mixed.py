#!/usr/bin/env python
"""Golden vectors of PPO on MIXED observations, produced by running the REAL reference (SurrealAI/surreal @ /root/reference)
with the stand-ins of ``_ref_harness.py`` and the helpers of ``make_golden.py``.  Run in the build container only:

    python tests/golden/make_golden_mixed.py      # writes tests/golden/ppo_learn_mixed_*.npz

  fixture               reference code that produced it
  --------------------  -----------------------------------------------------------------
  ppo_learn_mixed_*.npz surreal/learner/ppo.py:420-666 PPOLearner.learn / publish_parameter with a camera frame AND low-dim
                        inputs: z-filtered low-dim ++ CNN features into actor and critic (ppo_net.py:130-166,262-282)
"""
import copy
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from make_golden import H, PPOLearner, cfg_ppo, save, sd_np  # noqa: E402  (installs the reference harness)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def gen_ppo_learn_mixed():
    """Mixed observations (the default robosuite-style spec, ppo_configs.py:111-114): one uint8 frame through the shared CNN
    stem plus two low-dim inputs (widths 4 and 3: Dl = 7, not a multiple of 4) through the z-filter; actor and critic see
    cat([zfilter(low_dim), cnn_features], -1) (ppo_net.py:262-275).  The z-filter on (clip, adapt) and off (clip)."""
    C, HW, F = 2, 20, 12
    keys = (('robot-state', 4), ('object-state', 3))
    for tag, mode, use_z in (('mixed_clip', 'clip', True), ('mixed_adapt', 'adapt', True), ('mixed_clip_noz', 'clip', False)):
        torch.manual_seed(19)
        lc, ec, sc = cfg_ppo(mode=mode, B=6, n_step=4, stride=4, use_z=use_z, exp_interval=12)
        ec.obs_spec = {'low_dim': {k: (w,) for k, w in keys}, 'pixel': {'camera0': (C, HW, HW)}}
        ec.pixel_input = True
        lc.model.cnn_feature_dim = F
        L = H.construct_without_initialize(PPOLearner, lc, ec, sc)
        L._ps_publisher = H._Any()
        L.tensorplex = H._Any()
        L.ref_target_model.update_target_params(L.model)
        rng = np.random.default_rng(19)
        B, n, A = L.batch_size, L.n_step, 3
        out = dict(**sd_np(L.model, 'init/'))
        stats_all, hyper, captured = [], [], {}
        orig_opt, orig_gae = L._optimize, L._gae_and_return

        def opt_hook(*a, **k):
            st = orig_opt(*a, **k)
            captured['stats'] = {kk: float(vv) for kk, vv in st.items()}
            return st

        def gae_hook(*a, **k):
            adv, ret = orig_gae(*a, **k)
            captured['adv'], captured['ret'] = adv.detach().clone().numpy(), ret.detach().clone().numpy()
            return adv, ret
        L._optimize, L._gae_and_return = opt_hook, gae_hook

        def obs_dict(m):
            return {'pixel': {'camera0': rng.integers(0, 256, size=(B, m, C, HW, HW), dtype=np.uint8)},
                    'low_dim': {k: (rng.standard_normal((B, m, w)) * 1.5 + 0.3).astype(np.float32) for k, w in keys}}
        for it in range(2):
            obs, obs_next = obs_dict(n), obs_dict(1)
            with torch.no_grad():
                flat = {'pixel': {'camera0': torch.tensor(obs['pixel']['camera0'].reshape(B * n, C, HW, HW), dtype=torch.float32)},
                        'low_dim': {k: torch.tensor(obs['low_dim'][k].reshape(B * n, w)) for k, w in keys}}
                pd = L.model.forward_actor(flat).numpy().reshape(B, n, 2 * A)
            pd = pd.copy()
            pd[:, :, A:] *= np.exp(rng.uniform(-0.25, 0.25, size=(B, 1, 1))).astype(np.float32)
            actions = np.clip(rng.standard_normal((B, n, A)) * pd[:, :, A:] + pd[:, :, :A], -1, 1)
            rewards = rng.standard_normal((B, n)) * 0.5 + 0.1
            dones = np.zeros((B, n), dtype=np.float32)
            dones[rng.random(B) < 0.3, n - 1] = 1.0
            batch = H._AttrDict(obs=copy.deepcopy(obs), obs_next=copy.deepcopy(obs_next), actions=actions.copy(),
                                rewards=rewards.copy(), dones=dones.copy(), persistent_infos=[pd.astype(np.float32).copy()],
                                onetime_infos=None)
            for k, v in dict(actions=actions, rewards=rewards, dones=dones, pd=pd.astype(np.float32)).items():
                out['it%d/%s' % (it, k)] = v
            for name, o in (('obs', obs), ('obs_next', obs_next)):
                out['it%d/%s/pixel' % (it, name)] = o['pixel']['camera0']
                for k, _ in keys:
                    out['it%d/%s/%s' % (it, name, k)] = o['low_dim'][k]
            L.learn(batch)
            stats_all.append(captured['stats'])
            out['it%d/adv' % it], out['it%d/ret' % it] = captured['adv'], captured['ret']
            L.publish_parameter(it, message='')
            out.update(sd_np(L.model, 'it%d/after/' % it))
            hyper.append(dict(clip_epsilon=getattr(L, 'clip_epsilon', None), beta=getattr(L, 'beta', None),
                              exp_counter=L.exp_counter, kl_record=list(map(float, L.kl_record))))
        cfg = dict(mode=L.ppo_mode, B=B, n_step=n, A=A, C=C, HW=HW, cnn_feature_dim=F, low_dim=[list(kw) for kw in keys],
                   use_z_filter=use_z, actor_h=lc.model.actor_fc_hidden_sizes, critic_h=lc.model.critic_fc_hidden_sizes,
                   lr=lc.algo.network.lr_actor, exp_interval=lc.parameter_publish.exp_interval, iters=2)
        save('ppo_learn_' + tag, cfg=cfg, stats=stats_all, hyper=hyper, **out)


if __name__ == '__main__':
    gen_ppo_learn_mixed()
