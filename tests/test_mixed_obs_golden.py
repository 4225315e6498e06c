"""Mixed observations (a camera frame and low-dim inputs, the robosuite spec of ppo_configs.py:111-114) on the CPU:

  * the mixed oracle learner against goldens produced by the REAL reference's PPOLearner on that spec, with the z-filter on
    (clip, adapt) and off (clip);
  * the record layout of utils.obs_packed_dim / obs_layout: offsets, padding, packing, rejection of odd frame sizes."""
import numpy as np
import pytest
import torch

from oracle import nets
from oracle.filters import ZFilter
from oracle.ppo_mixed import OraclePPOLearnerMixed
from surreal_b200 import utils as U

torch.set_num_threads(1)
T = torch.tensor


def mixed_batch(b, keys):
    """golden per-iteration arrays -> aggregator-format batch dict with mixed observation dicts (numpy, host)."""
    def obs(name):
        return {'pixel': {'camera0': b['%s/pixel' % name]}, 'low_dim': {k: b['%s/%s' % (name, k)] for k, _ in keys}}
    return {'obs': obs('obs'), 'obs_next': obs('obs_next'), 'actions': b['actions'], 'rewards': b['rewards'],
            'dones': b['dones'], 'persistent_infos': [b['pd']], 'onetime_infos': None, 'pd': b['pd']}


def mixed_oracle(g):
    cfg = g.js('cfg')
    init = g.sub('init/')
    actor = nets.params_from_state(init, 'actor/model/')
    critic = nets.params_from_state(init, 'critic/model/')
    zf = None
    if 'z_filter/count' in init:
        zf = ZFilter(len(init['z_filter/running_sum'])).load(init['z_filter/running_sum'], init['z_filter/running_sumsq'],
                                                             init['z_filter/count'])
    conv = [(T(init['cnn_stem/model/seq/%d/weight' % i]), T(init['cnn_stem/model/seq/%d/bias' % i])) for i in (0, 2)]
    fc = (T(init['cnn_stem/model/seq/5/weight']), T(init['cnn_stem/model/seq/5/bias']))
    return OraclePPOLearnerMixed(actor, T(init['actor/log_var']), critic, zf, conv, [4, 2], fc,
                                 (cfg['C'], cfg['HW'], cfg['HW']), cfg['A'], cfg['n_step'], cfg['B'], ppo_mode=cfg['mode'],
                                 lr_actor=cfg['lr'], lr_critic=cfg['lr'], exp_interval=cfg['exp_interval'])


@pytest.mark.parametrize('tag', ['mixed_clip', 'mixed_adapt', 'mixed_clip_noz'])
def test_ppo_learn_mixed_oracle(golden, tag):
    g = golden('ppo_learn_' + tag)
    cfg, hyper, stats = g.js('cfg'), g.js('hyper'), g.js('stats')
    assert ('z_filter/count' in g.sub('init/')) == cfg['use_z_filter']
    L = mixed_oracle(g)
    F = cfg['cnn_feature_dim']
    Dl = sum(w for _, w in cfg['low_dim'])
    assert L.actor[0][0].shape[1] == Dl + F                     # layer 0 takes [low-dim | features]
    for it in range(cfg['iters']):
        b = g.sub('it%d/' % it)
        assert b['obs/pixel'].dtype == np.uint8
        st = L.learn(mixed_batch(b, cfg['low_dim']))
        np.testing.assert_allclose(L.last_adv.numpy(), b['adv'], rtol=0, atol=2e-6)
        np.testing.assert_allclose(L.last_ret.numpy(), b['ret'], rtol=0, atol=2e-6)
        L.publish_parameter()
        for k, v in stats[it].items():
            assert st[k] == pytest.approx(v, rel=1e-5, abs=1e-6), k
        after = g.sub('it%d/after/' % it)
        for i, (w, bb) in zip((0, 2), L.conv):
            np.testing.assert_allclose(w.detach().numpy(), after['cnn_stem/model/seq/%d/weight' % i], rtol=0, atol=1e-6)
            np.testing.assert_allclose(bb.detach().numpy(), after['cnn_stem/model/seq/%d/bias' % i], rtol=0, atol=1e-6)
        np.testing.assert_allclose(L.fc[0].detach().numpy(), after['cnn_stem/model/seq/5/weight'], rtol=0, atol=1e-6)
        for i, (w, bb) in enumerate(L.actor):
            np.testing.assert_allclose(w.detach().numpy(), after['actor/model/seq/%d/weight' % (2 * i)], rtol=0, atol=1e-6)
        for i, (w, bb) in enumerate(L.critic):
            np.testing.assert_allclose(w.detach().numpy(), after['critic/model/seq/%d/weight' % (2 * i)], rtol=0, atol=1e-6)
        if cfg['use_z_filter']:
            for k in ('running_sum', 'running_sumsq', 'count'):
                np.testing.assert_allclose(getattr(L.zf.zf, k).numpy().reshape(-1), after['z_filter/' + k].reshape(-1),
                                           rtol=1e-6, atol=0, err_msg=k)
        if cfg['mode'] == 'clip':
            assert L.clip_epsilon == pytest.approx(hyper[it]['clip_epsilon'], rel=1e-12)
        else:
            assert L.beta == pytest.approx(hyper[it]['beta'], rel=1e-12)


SPEC = {'low_dim': {'robot-state': (4,), 'object-state': (3,)}, 'pixel': {'camera0': (2, 20, 20)}}


def test_mixed_record_layout():
    lay = U.obs_layout(SPEC)
    assert U.obs_is_mixed(SPEC) and U.obs_is_pixel(SPEC)
    assert lay['frame_bytes'] == 800 and lay['low_dim_off'] == 200 and lay['low_dim'] == 7
    assert lay['keys'] == [('robot-state', 200, 4), ('object-state', 204, 3)]
    assert lay['width'] == 208 == U.obs_packed_dim(SPEC)           # 207 words padded to a multiple of 4
    # 4x84x84 frame + 32 low-dim floats: no padding needed; + 1 float: 12 bytes of padding
    assert U.obs_packed_dim({'pixel': {'camera0': (4, 84, 84)}, 'low_dim': {'s': (32,)}}) == 7056 + 32
    assert U.obs_packed_dim({'pixel': {'camera0': (4, 84, 84)}, 'low_dim': {'s': (33,)}}) == 7056 + 36
    for spec in ({'low_dim': {'s': (3,)}, 'pixel': {'camera0': (1, 3, 3)}}, {'pixel': {'camera0': (3, 5, 5)}}):
        with pytest.raises(ValueError, match='multiple of 16 bytes'):
            U.obs_packed_dim(spec)


def test_single_kind_layouts_unchanged():
    assert U.obs_packed_dim({'low_dim': {'a': (5,), 'b': (6,)}}) == 11
    assert U.obs_packed_dim({'pixel': {'camera0': (4, 84, 84)}}) == 7056
    assert U.obs_packed_dim({'pixel': {'camera0': (4, 84, 84)}, 'low_dim': {}}) == 7056
    assert not U.obs_is_mixed({'pixel': {'camera0': (4, 84, 84)}})


def test_pack_obs_rows_round_trip():
    lay = U.obs_layout(SPEC)
    rng = np.random.default_rng(3)
    obs = {'pixel': {'camera0': rng.integers(0, 256, (5, 2, 2, 20, 20), dtype=np.uint8)},
           'low_dim': {'robot-state': rng.standard_normal((5, 2, 4)).astype(np.float32),
                       'object-state': rng.standard_normal((5, 2, 3)).astype(np.float32)}}
    rows = U.pack_obs_rows(obs, lay)
    assert rows.shape == (5, 2, 208) and rows.dtype == np.float32
    assert np.array_equal(rows[..., :200].copy().view(np.uint8).reshape(5, 2, 2, 20, 20), obs['pixel']['camera0'])
    assert np.array_equal(rows[..., 200:204], obs['low_dim']['robot-state'])
    assert np.array_equal(rows[..., 204:207], obs['low_dim']['object-state'])
    assert not rows[..., 207:].any()
    flat = U.obs_flat({'pixel': {'camera0': obs['pixel']['camera0'][:, 0]},
                       'low_dim': {k: v[:, 0] for k, v in obs['low_dim'].items()}}, SPEC)
    assert np.array_equal(flat.view(np.uint32), rows[:, 0].copy().view(np.uint32))     # frame words may read as NaN
    views = U.mixed_obs_views(torch.from_numpy(rows), lay)
    assert torch.equal(views['pixel']['camera0'], torch.from_numpy(obs['pixel']['camera0']))
    for k in obs['low_dim']:
        assert torch.equal(views['low_dim'][k], torch.from_numpy(obs['low_dim'][k]))
