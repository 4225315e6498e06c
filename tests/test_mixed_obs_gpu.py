"""Mixed observations on the GPU: one uint8 camera frame plus low-dim inputs (the robosuite spec, ppo_configs.py:111-114).
The CNN stem reads the frames and the heads read the low-dim columns in place from the packed record rows
(utils.obs_layout); actor and critic see cat([zfilter(low_dim), cnn_features], -1) (ppo_net.py:262-275).

  * PPOLearner.learn + publish against goldens produced by the REFERENCE's PPOLearner on that spec (z-filter on and off);
  * device mixed env -> PPOAgent.act -> window staging -> HBM FIFO -> learn(), against the mixed oracle;
  * the same record identity through a host numpy env;
  * the strided conv-1 entry points against the contiguous ones;
  * reference-keyed state dicts load into learner and agent; mixed + data parallel raises."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import ppo_configs, ref_state_dict
from test_mixed_obs_golden import mixed_batch

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'

LOSS_STATS = ['_surr_loss', '_clip_surr_loss', '_kl_loss_adapt', '_entropy', '_pol_kl', '_val_loss', '_avg_return_targ',
              '_avg_log_sig', '_avg_behave_likelihood', '_avg_is_weight', '_ref_behave_diff']
KEYS = (('robot-state', 4), ('object-state', 3))


def _mixed_cfg(C_, HW, F, A, actor_h, critic_h, n, B, mode, lr, exp_interval, keys=KEYS, use_z=True, N=None):
    lc, ec, sc = ppo_configs(D=1, A=A, actor_h=actor_h, critic_h=critic_h, n_step=n, stride=n, B=B, mode=mode, lr=lr,
                             exp_interval=exp_interval, use_z=use_z)
    ec.obs_spec = {'low_dim': {k: (w,) for k, w in keys}, 'pixel': {'camera0': (C_, HW, HW)}}
    ec.pixel_input = True
    lc.model.cnn_feature_dim = F
    if N is not None:
        ec.num_envs = N
    return lc, ec, sc


def _golden_cfg(cfg):
    return _mixed_cfg(cfg['C'], cfg['HW'], cfg['cnn_feature_dim'], cfg['A'], cfg['actor_h'], cfg['critic_h'], cfg['n_step'],
                      cfg['B'], cfg['mode'], cfg['lr'], cfg['exp_interval'], keys=[tuple(kw) for kw in cfg['low_dim']],
                      use_z=cfg['use_z_filter'])


def _assert_zfilter(model, ref_sd):
    got = model.state_dict()
    for k in ('z_filter.running_sum', 'z_filter.running_sumsq', 'z_filter.count'):
        e = ref_sd[k].reshape(-1).double()
        assert float((got[k].cpu().reshape(-1).double() - e).abs().max()) <= 1e-6 * max(1.0, float(e.abs().max())), k


@pytest.mark.parametrize('tag', ['mixed_clip', 'mixed_adapt', 'mixed_clip_noz'])
def test_ppo_learn_mixed_matches_reference(golden, tag):
    from surreal_b200.learner import PPOLearner
    g = golden('ppo_learn_' + tag)
    cfg, hyper, stats = g.js('cfg'), g.js('hyper'), g.js('stats')
    L = PPOLearner(*_golden_cfg(cfg))
    assert L.mixed
    L.model.load_state_dict(ref_state_dict(g.sub('init/')))
    L.ref_target_model.update_target_params(L.model)
    lr = cfg['lr']
    for it in range(cfg['iters']):
        b = g.sub('it%d/' % it)
        st = L.learn(mixed_batch(b, cfg['low_dim']))
        L.publish_parameter(it, message='')
        torch.cuda.synchronize()
        assert float((L._adv.cpu() - torch.tensor(b['adv'])).abs().max()) <= 1e-5
        rms = float(np.sqrt((b['ret'] ** 2).mean()))
        assert float((L._ret.cpu() - torch.tensor(b['ret'])).abs().max()) <= 1e-5 * max(1.0, rms)
        for k, v in stats[it].items():
            assert k in st, k
            tol = 1e-5 * max(1.0, abs(v)) if k in LOSS_STATS else 2e-4 * max(1.0, abs(v))
            if k == '_val_explained_var':
                tol = 1e-4
            assert abs(st[k] - v) <= tol, '%s it%d: got %.9g expected %.9g' % (k, it, st[k], v)
        after = ref_state_dict(g.sub('it%d/after/' % it))
        got = L.model.state_dict()
        assert set(after) == set(got), sorted(set(after) ^ set(got))
        worst = 0.0
        for k, e in after.items():
            if not k.startswith('z_filter.'):
                worst = max(worst, float((got[k].cpu().reshape(e.shape) - e).abs().max()))
        assert worst <= max(2e-6, 0.02 * lr), 'params drifted by %.3e' % worst
        if cfg['use_z_filter']:
            _assert_zfilter(L.model, after)
        if cfg['mode'] == 'clip':
            assert L.clip_epsilon == pytest.approx(hyper[it]['clip_epsilon'], rel=1e-12)
        else:
            assert L.beta == pytest.approx(hyper[it]['beta'], rel=1e-12)


def _seed_zfilter(model, rng):
    """Non-trivial z-filter statistics (fresh ones only clamp), loaded through the reference keys."""
    sd = model.state_dict()
    D = sd['z_filter.running_sum'].numel()
    cnt = 50.0
    mean = rng.standard_normal(D) * 0.3
    var = rng.uniform(0.2, 2.0, D)
    sd['z_filter.running_sum'] = torch.tensor(mean * cnt, dtype=torch.float32)
    sd['z_filter.running_sumsq'] = torch.tensor((var + mean ** 2) * cnt, dtype=torch.float32)
    sd['z_filter.count'] = torch.tensor([cnt], dtype=torch.float32)
    model.load_state_dict(sd)
    return sd


def _oracle_from(sd, frame_shape, A, n, B, keys_dl):
    from oracle.filters import ZFilter
    from oracle.ppo_mixed import OraclePPOLearnerMixed
    sd = {k: v.cpu() for k, v in sd.items()}
    conv = [(sd['cnn_stem.model.seq.%d.weight' % i], sd['cnn_stem.model.seq.%d.bias' % i]) for i in (0, 2)]
    fc = (sd['cnn_stem.model.seq.5.weight'], sd['cnn_stem.model.seq.5.bias'])
    al = [(sd['actor.model.seq.%d.weight' % (2 * i)], sd['actor.model.seq.%d.bias' % (2 * i)]) for i in range(3)]
    cl = [(sd['critic.model.seq.%d.weight' % (2 * i)], sd['critic.model.seq.%d.bias' % (2 * i)]) for i in range(3)]
    zf = ZFilter(keys_dl).load(sd['z_filter.running_sum'], sd['z_filter.running_sumsq'], sd['z_filter.count'])
    return OraclePPOLearnerMixed(al, sd['actor.log_var'].view(1, A), cl, zf, conv, [4, 2], fc, frame_shape, A, n, B,
                                 ppo_mode='clip', lr_actor=1e-4, lr_critic=1e-4, exp_interval=B)


def _check_batch_against_oracle(batch, ag, lc, ec, sc, noise, N, n, A, frame_shape):
    """pd rows == oracle stem || z-filtered low-dim -> actor on the staged observations; learn() == the mixed oracle."""
    from surreal_b200.learner import PPOLearner
    Dl = sum(w for _, w in KEYS)
    sd = ag.model.state_dict()
    O = _oracle_from(sd, frame_shape, A, n, N, Dl)
    host = lambda o: {'pixel': {'camera0': o['pixel']['camera0'].cpu().numpy()},  # noqa: E731
                      'low_dim': {k: o['low_dim'][k].cpu().numpy() for k, _ in KEYS}}
    hobs, hobs_next = host(batch['obs']), host(batch['obs_next'])
    with torch.no_grad():
        x = torch.tensor(O.flat(hobs)).reshape(N * n, -1)
        mean = O.forward_actor(x)[:, :A]
    pd = batch['persistent_infos'][0].cpu().view(N * n, 2 * A)
    assert float((pd[:, :A] - mean).abs().max()) <= 1e-5
    std = torch.exp(sd['actor.log_var'].cpu()).view(1, A) * \
        torch.exp(torch.tensor(noise, dtype=torch.float32)).repeat_interleave(n).view(-1, 1)
    assert float((pd[:, A:] - std).abs().max()) <= 1e-6
    L = PPOLearner(lc, ec, sc)
    L.model.load_state_dict(sd)
    L.ref_target_model.update_target_params(L.model)
    st_o = O.learn(dict(obs=hobs, obs_next=hobs_next, actions=batch['actions'].cpu().numpy(),
                        rewards=batch['rewards'].cpu().numpy(), dones=batch['dones'].cpu().numpy(),
                        pd=batch['persistent_infos'][0].cpu().numpy()))
    st = L.learn(batch)
    torch.cuda.synchronize()
    assert L.last_n_policy_epochs == O.n_policy_epochs[-1]
    for k in ('_surr_loss', '_clip_surr_loss', '_pol_kl', '_val_loss', '_entropy', '_avg_return_targ', '_avg_is_weight',
              'obs_running_mean', 'obs_running_std'):
        assert abs(st[k] - st_o[k]) <= 1e-5 * max(1.0, abs(st_o[k])), (k, st[k], st_o[k])
    assert float((L._adv.cpu().view(-1) - O.last_adv.view(-1)).abs().max()) <= 1e-5
    zs = L.model.state_dict()
    assert float((zs['z_filter.running_sum'].cpu() - O.zf.zf.running_sum).abs().max()) <= 1e-4
    assert float(zs['z_filter.count'].cpu()[0]) == float(O.zf.zf.count[0])


def _records_equal(batch, seen, n):
    fr = torch.cat([batch['obs']['pixel']['camera0'], batch['obs_next']['pixel']['camera0']], 1)
    assert fr.dtype == torch.uint8
    for t in range(n + 1):
        assert torch.equal(fr[:, t].cpu(), seen[t]['pixel']), 'frame %d changed on the way through staging / replay' % t
        for k, _ in KEYS:
            lo = torch.cat([batch['obs']['low_dim'][k], batch['obs_next']['low_dim'][k]], 1)
            assert torch.equal(lo[:, t].cpu().view(torch.int32), seen[t][k].view(torch.int32)), (k, t)


def test_mixed_actors_replay_learner_end_to_end():
    """Device mixed env -> PPOAgent.act (stem + head with z-filter and aux features + sampling) -> window staging -> HBM FIFO
    -> PPOLearner.learn: frames and low-dim rows bit-identical, pd rows and learn() equal to the mixed oracle."""
    from surreal_b200.agent import PPOAgent
    from surreal_b200.replay import FIFOReplay
    from surreal_b200.env import SyntheticMixedEnv
    N, C_, HW, Fd, A, n = 16, 4, 28, 24, 3, 5
    lc, ec, sc = _mixed_cfg(C_, HW, Fd, A, (32, 24), (28, 20), n, N, 'clip', 1e-4, N, N=N)
    lc.replay.memory_size = 4 * N
    ec.env_name = 'synthetic'
    R = FIFOReplay(lc, ec, sc)
    ag = PPOAgent(lc, ec, sc, 0, 'training')
    noise = np.linspace(-0.2, 0.2, N)
    ag.set_noise(noise)
    _seed_zfilter(ag.model, np.random.default_rng(4))
    assert isinstance(ag.get_env(), SyntheticMixedEnv)        # the env an Agent builds for a mixed spec
    env = SyntheticMixedEnv(N, ec.obs_spec, A, limit_episode_length=2 * n, seed=5)
    ag.env = w = ag.prepare_env_agent(env)
    snap = lambda o: dict(pixel=o['pixel']['camera0'].cpu().clone(),  # noqa: E731
                          **{k: o['low_dim'][k].cpu().clone() for k, _ in KEYS})
    obs, _ = w.reset()
    seen = [snap(obs)]
    for _ in range(n):
        a = ag.act(obs)
        obs, _, _, info = w.step(a)
        seen.append(snap(info['obs_next']))
    torch.cuda.synchronize()
    assert len(R) == N
    batch = R.sample(N)
    _records_equal(batch, seen, n)
    _check_batch_against_oracle(batch, ag, lc, ec, sc, noise, N, n, A, (C_, HW, HW))


def test_mixed_env_matches_pixel_and_lowdim_envs():
    """SyntheticMixedEnv = SyntheticPixelEnv's frames + SyntheticEnv's low-dim dynamics, reward and done (same seed)."""
    from surreal_b200.env import SyntheticEnv, SyntheticPixelEnv, SyntheticMixedEnv
    N, A, shape = 8, 3, (4, 12, 12)
    spec = {'pixel': {'camera0': shape}, 'low_dim': {'s': (9,)}}
    M, P, E = SyntheticMixedEnv(N, spec, A, 3, seed=2), SyntheticPixelEnv(N, shape, A, 3, seed=2), SyntheticEnv(N, 9, A, 3, seed=2)
    om, _ = M.reset()
    P.reset()
    E.reset()
    P.state.copy_(om['pixel']['camera0'].reshape(N, -1))
    E.state.copy_(om['low_dim']['s'])
    g = torch.Generator().manual_seed(0)
    for _ in range(5):
        a = (torch.rand(N, A, generator=g) * 2 - 1).to(DEV)
        om, rm, dm, im = M.step(a)
        op, _, dp, ip = P.step(a)
        oe, re, de, ie = E.step(a)
        for c in (M, P, E):
            c.step_counter += 1
        assert torch.equal(om['pixel']['camera0'], op['pixel']['camera0'])
        assert torch.equal(im['obs_next']['pixel']['camera0'], ip['obs_next']['pixel']['camera0'])
        assert torch.equal(om['low_dim']['s'], oe['low_dim']['flat_inputs'])
        assert torch.equal(im['obs_next']['low_dim']['s'], ie['obs_next'])
        assert torch.equal(rm, re) and torch.equal(dm, de) and torch.equal(dm, dp)


class _HostMixedEnv:
    """A batched host env (numpy in / out) with a frame and two low-dim keys, like a robosuite vector env."""

    def __init__(self, N, spec, A, seed):
        self.N, self.A, self.spec = N, A, spec
        self.rng = np.random.default_rng(seed)

    def observation_spec(self):
        return self.spec

    def _draw(self):
        return {'pixel': {'camera0': self.rng.integers(0, 256, (self.N,) + tuple(self.spec['pixel']['camera0']), dtype=np.uint8)},
                'low_dim': {k: self.rng.standard_normal((self.N,) + tuple(v)).astype(np.float32)
                            for k, v in self.spec['low_dim'].items()}}

    def reset(self):
        return self._draw(), {}

    def step(self, action):
        a = action[0] if isinstance(action, tuple) else action
        assert isinstance(a, np.ndarray) and a.shape == (self.N, self.A)
        return self._draw(), self.rng.standard_normal(self.N).astype(np.float32), np.zeros(self.N, np.float32), {}


def test_mixed_host_env_records():
    """Host numpy dicts (frame + two low-dim keys) -> PPOAgent.act (packed into a pinned row) -> host window staging -> FIFO:
    the records equal what the env produced, bit for bit, and learn() equals the mixed oracle."""
    from surreal_b200.agent import PPOAgent
    from surreal_b200.replay import FIFOReplay
    N, C_, HW, Fd, A, n = 8, 2, 20, 12, 3, 4
    lc, ec, sc = _mixed_cfg(C_, HW, Fd, A, (32, 24), (28, 20), n, N, 'clip', 1e-4, N, N=N)
    lc.replay.memory_size = 4 * N
    R = FIFOReplay(lc, ec, sc)
    ag = PPOAgent(lc, ec, sc, 0, 'training')
    noise = np.linspace(-0.1, 0.1, N)
    ag.set_noise(noise)
    _seed_zfilter(ag.model, np.random.default_rng(6))
    ag.env = w = ag.prepare_env_agent(_HostMixedEnv(N, ec.obs_spec, A, seed=8))
    snap = lambda o: dict(pixel=torch.from_numpy(o['pixel']['camera0'].copy()),  # noqa: E731
                          **{k: torch.from_numpy(o['low_dim'][k].copy()) for k, _ in KEYS})
    obs, _ = w.reset()
    seen = [snap(obs)]
    for _ in range(n):
        a = ag.act(obs)
        assert isinstance(a[0], np.ndarray)
        obs, _, _, _ = w.step(a)
        seen.append(snap(obs))
    torch.cuda.synchronize()
    assert len(R) == N
    batch = R.sample(N)
    _records_equal(batch, seen, n)
    _check_batch_against_oracle(batch, ag, lc, ec, sc, noise, N, n, A, (C_, HW, HW))


def test_conv1_strided_entry_points_bitwise():
    """Frames read in place from wider rows give the same bits as the contiguous conv-1 forward and weight gradient."""
    from surreal_b200 import _lib, ops
    from surreal_b200.model.cnn_stem import CNNStem
    L, st = _lib.lib(), ops._stream()
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    Cc, H, W, R = 4, 36, 36, 37
    fb = Cc * H * W
    rb = fb + 4 * 13                                             # row stride > frame size (odd word count of padding)
    g = torch.Generator().manual_seed(11)
    frames = torch.randint(0, 256, (R, Cc, H, W), generator=g, dtype=torch.uint8).to(DEV)
    rows = torch.randint(0, 256, (R, rb), generator=g, dtype=torch.uint8).to(DEV)
    rows[:, :fb].copy_(frames.view(R, -1))
    stem = CNNStem((Cc, H, W), 8, DEV)
    w1, b1 = stem.seg('w1'), stem.seg('b1')
    y0 = torch.zeros(R, 16, stem.H1, stem.W1, device=DEV)
    y1 = torch.full_like(y0, 7.0)
    _lib.check(L.sb200_conv_forward_f32(1, p(frames), 1, R, Cc, H, W, p(w1), p(b1), 1.0 / 255.0, p(y0), st), 'fwd')
    _lib.check(L.sb200_conv1_forward_u8_strided(p(rows), rb, R, Cc, H, W, p(w1), p(b1), 1.0 / 255.0, p(y1), st), 'fwd strided')
    torch.cuda.synchronize()
    assert torch.equal(y0, y1) and float(y0.abs().sum()) > 0
    dy = torch.randn(R, 16, stem.H1, stem.W1, generator=g).to(DEV)
    splits = 5
    n1 = w1.numel() + 16
    s0 = torch.zeros(splits, n1 + 16, device=DEV)
    s1 = torch.full_like(s0, 3.0)
    for buf, fn in ((s0, lambda s: L.sb200_conv_backward_dw_f32(1, p(frames), 1, p(dy), R, Cc, H, W, 1.0 / 255.0, p(s),
                                                              C.c_void_p(s.data_ptr() + 4 * w1.numel()), s.shape[1], splits, st)),
                    (s1, lambda s: L.sb200_conv1_backward_dw_u8_strided(p(rows), rb, p(dy), R, Cc, H, W, 1.0 / 255.0, p(s),
                                                                      C.c_void_p(s.data_ptr() + 4 * w1.numel()), s.shape[1],
                                                                      splits, st))):
        _lib.check(fn(buf), 'dw')
    torch.cuda.synchronize()
    assert torch.equal(s0[:, :n1], s1[:, :n1]) and float(s0[:, :n1].abs().sum()) > 0


def test_reference_state_dict_loads_into_learner_and_agent(golden):
    """A reference-written mixed-mode state dict (the golden's init, keys of pixel mode + z_filter.*) loads into the learner
    and into the agent; both forward like the reference (the golden's behaviour means), and data parallel is refused."""
    from surreal_b200.learner import PPOLearner
    from surreal_b200.agent import PPOAgent
    g = golden('ppo_learn_mixed_clip')
    cfg = g.js('cfg')
    lc, ec, sc = _golden_cfg(cfg)
    sd = ref_state_dict(g.sub('init/'))
    L = PPOLearner(lc, ec, sc)
    assert set(L.model.state_dict()) == set(sd)
    L.model.load_state_dict(sd)
    ec.num_envs = cfg['B'] * cfg['n_step']
    ag = PPOAgent(lc, ec, sc, 0, 'eval_deterministic_local')
    ag.model.load_state_dict(sd)
    b = g.sub('it0/')
    B, n, A = cfg['B'], cfg['n_step'], cfg['A']
    obs = {'pixel': {'camera0': torch.tensor(b['obs/pixel']).reshape(B * n, cfg['C'], cfg['HW'], cfg['HW']).to(DEV)},
           'low_dim': {k: torch.tensor(b['obs/' + k]).reshape(B * n, -1).to(DEV) for k, _ in cfg['low_dim']}}
    pd_l = L.model.forward_actor(obs).cpu()
    pd_a = ag.model.forward_actor(obs).cpu()
    assert torch.equal(pd_l, pd_a)
    want = torch.tensor(b['pd']).reshape(B * n, 2 * A)[:, :A]
    assert float((pd_l[:, :A] - want).abs().max()) <= 1e-5
    host = {'pixel': {'camera0': b['obs/pixel'].reshape(B * n, cfg['C'], cfg['HW'], cfg['HW'])},
            'low_dim': {k: b['obs/' + k].reshape(B * n, -1) for k, _ in cfg['low_dim']}}
    act = ag.act(host)                                            # deterministic: the mean, through the packed-row path
    assert isinstance(act, np.ndarray)
    assert float(np.abs(act - pd_l[:, :A].numpy()).max()) <= 1e-6
    with pytest.raises(NotImplementedError, match='mixed'):
        L.enable_data_parallel()
