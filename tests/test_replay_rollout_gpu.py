"""HBM replay, device-side experience windowing and batched actors vs the reference-generated goldens
and the CPU oracle.  Bit-exact for indices / ordering / slot assignment."""
import random

import numpy as np
import pytest
import torch

from helpers import ppo_configs, ddpg_configs, ref_state_dict
from oracle.windowing import multistep_windows, ssar_nstep
from oracle.replay import FIFO as OFIFO

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _window(i, n, D, A):
    """a host window whose every field encodes the id i"""
    ob = lambda v: {'low_dim': {'flat_inputs': np.full((D,), v, dtype=np.float32)}}  # noqa: E731
    return dict(obs=[ob(i + 0.001 * k) for k in range(n)], obs_next=ob(i + 0.5),
                actions=[np.full((A,), i, dtype=np.float64) for _ in range(n)], rewards=[float(i)] * n,
                dones=[False] * (n - 1) + [True], persistent_infos=[[np.full((2 * A,), i, dtype=np.float32)]] * n,
                onetime_infos=[], infos=[{}] * n, n_step=n)


def test_fifo_replay_trace_matches_reference(golden):
    from surreal_b200.replay import FIFOReplay
    f = golden('replay').js('fifo')
    n, D, A = 3, 5, 2
    lc, ec, sc = ppo_configs(D=D, A=A, n_step=n, stride=n, B=f['batch_size'], memory_size=f['memory_size'])
    R = FIFOReplay(lc, ec, sc)
    nxt = 0
    for (op, k), tr in zip(f['script'], f['trace']):
        if op == 'insert':
            for _ in range(k):
                R.insert(_window(nxt, n, D, A))
                nxt += 1
            assert [len(R), int(R.start_sample_condition())] == tr
        else:
            b = R.sample(k)
            ids = b['rewards'][:, 0].cpu().numpy().astype(int).tolist()
            assert ids == tr
            assert b['obs']['low_dim']['flat_inputs'].shape == (k, n, D)
            assert torch.allclose(b['obs_next']['low_dim']['flat_inputs'][:, 0, 0].cpu(), torch.tensor(tr, dtype=torch.float32) + 0.5)
            assert b['persistent_infos'][0][:, 0, 0].cpu().numpy().astype(int).tolist() == tr
            assert bool((b['dones'][:, -1] == 1).all()) and bool((b['dones'][:, 0] == 0).all())
    with pytest.raises(IndexError):
        while True:
            R.sample(f['batch_size'])


def test_uniform_replay_trace_matches_reference(golden):
    from surreal_b200.replay import UniformReplay
    u = golden('replay').js('uniform')
    D, A = 4, 2
    lc, ec, sc = ddpg_configs(D=D, A=A, B=8, memory_size=u['memory_size'], start=u['sampling_start_size'])
    R = UniformReplay(lc, ec, sc)
    random.seed(u['seed'])
    nxt = 0
    ob = lambda v: {'low_dim': {'flat_inputs': np.full((D,), v, dtype=np.float32)}}  # noqa: E731
    for (op, k), tr in zip(u['script'], u['trace']):
        if op == 'insert':
            for _ in range(k):
                R.insert({'obs': [ob(nxt), ob(nxt + 0.5)], 'action': np.full((A,), nxt / 1000.0), 'reward': float(nxt),
                          'done': nxt % 2 == 0, 'info': {}})
                nxt += 1
            assert [len(R), int(R.start_sample_condition()), R._host_next] == tr
        else:
            b = R.sample(k)
            assert b['rewards'][:, 0].cpu().numpy().astype(int).tolist() == tr
            assert b['obs']['low_dim']['flat_inputs'][:, 0].cpu().numpy().astype(int).tolist() == tr
            assert b['rewards'].shape == (k, 1) and b['dones'].shape == (k, 1)
            assert b['dones'][:, 0].cpu().numpy().astype(int).tolist() == [int(t % 2 == 0) for t in tr]


class ScriptedEnv:
    """Deterministic device env: obs = global step id of that actor, reward = 0.25*g - 3, scripted episode ends."""
    metadata = {}

    def __init__(self, scripts, D=2, A=1):
        self.scripts = [list(s) for s in scripts]
        self.N, self.D, self.A = len(scripts), D, A
        self.device = torch.device(DEV)
        self.step_counter = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.ep = [0] * self.N
        self.t = [0] * self.N
        self.g = [0] * self.N

    def _obs(self):
        return torch.tensor([[float(g)] * self.D for g in self.g], device=self.device)

    def reset(self):
        return {'low_dim': {'flat_inputs': self._obs()}}, {}

    def step(self, action):
        rew, done = [], []
        for i in range(self.N):
            self.t[i] += 1
            self.g[i] += 1
            rew.append(0.25 * self.g[i] - 3.0)
            done.append(float(self.t[i] >= self.scripts[i][self.ep[i] % len(self.scripts[i])]))
        obs_next = self._obs()
        for i in range(self.N):
            if done[i]:
                self.ep[i] += 1
                self.t[i] = 0
        return ({'low_dim': {'flat_inputs': obs_next.clone()}}, torch.tensor(rew, device=self.device),
                torch.tensor(done, device=self.device), {'obs_next': obs_next})


@pytest.mark.parametrize('case_id', [0, 1, 2, 3])
def test_window_staging_matches_reference_wrapper(golden, case_id):
    """One actor, the exact scripts of the golden: windows (obs ids, obs_next, dones, action/pd/reward payload)."""
    from surreal_b200.replay import FIFOReplay
    from surreal_b200.env import ExpSenderWrapperMultiStepMovingWindowWithInfo as W
    case = golden('window_multistep').js('cases')[case_id]
    n, stride, ep_lens = case['n_step'], case['stride'], case['ep_lens']
    lc, ec, sc = ppo_configs(D=2, A=1, n_step=n, stride=stride, B=1, memory_size=64)
    R = FIFOReplay(lc, ec, sc)
    env = ScriptedEnv([ep_lens])
    w = W(env, lc, sc, replay=R)
    w.reset()
    for _ in range(sum(ep_lens)):
        g = env.g[0]
        p = int(w.stage_pos[0].item())
        w.stage_act[0, p, 0] = float(g)                  # what sb200_ppo_sample_f32 stages for this step
        w.stage_pd[0, p, 0] = float(g)
        w.stage_pd[0, p, 1] = 1.0
        w.step(torch.zeros(1, 1, device=DEV))
    exp = case['windows']
    assert len(R) == len(exp)
    for e in exp:
        b = R.sample(1)
        assert b['obs']['low_dim']['flat_inputs'][0, :, 0].cpu().numpy().astype(int).tolist() == e['obs']
        assert int(b['obs_next']['low_dim']['flat_inputs'][0, 0, 0].item()) == e['obs_next']
        assert b['dones'][0].cpu().numpy().astype(bool).tolist() == e['dones']
        assert b['actions'][0, :, 0].cpu().numpy().tolist() == e['actions']
        assert b['persistent_infos'][0][0, :, 0].cpu().numpy().tolist() == e['pd0']
        np.testing.assert_allclose(b['rewards'][0].cpu().numpy(), np.array(e['rewards'], dtype=np.float32), rtol=0, atol=0)


def test_window_staging_many_actors_order_and_drop():
    """Several actors with different episode scripts: arrival order is (step, actor); FIFO drops the oldest."""
    from surreal_b200.replay import FIFOReplay
    from surreal_b200.env import ExpSenderWrapperMultiStepMovingWindowWithInfo as W
    n, stride = 4, 3
    scripts = [[9, 5], [4, 11], [7], [6, 6, 2], [13]]
    steps = 40
    lc, ec, sc = ppo_configs(D=2, A=1, n_step=n, stride=stride, B=2, memory_size=12)
    R = FIFOReplay(lc, ec, sc)
    env = ScriptedEnv(scripts)
    w = W(env, lc, sc, replay=R)
    w.reset()
    for _ in range(steps):
        w.step(torch.zeros(len(scripts), 1, device=DEV))
    # oracle: per-actor windows with their completion step, merged in (step, actor) order into a deque(maxlen=cap)
    events = []
    for a, sc_ in enumerate(scripts):
        ep_lens, tot = [], 0
        while tot < steps:
            L = sc_[len(ep_lens) % len(sc_)]
            ep_lens.append(min(L, steps - tot))
            tot += L
        # a truncated last episode must not emit a fake 'done'; only windows fully inside `steps` count
        for obs_ids, nxt, dones in multistep_windows(ep_lens, n, stride):
            if nxt <= steps:
                events.append((nxt, a, obs_ids))
    events.sort(key=lambda e: (e[0], e[1]))
    q = OFIFO(12, 2)
    for e in events:
        q.insert(e)
    st = R._read_state()
    assert st['count'] == len(q) and st['total_in'] == len(events) and st['dropped'] == len(events) - len(q)
    expect = list(q.q)
    ids = []
    for _ in range(len(q)):
        got = R.sample(1)
        ids.append(got['obs']['low_dim']['flat_inputs'][0, :, 0].cpu().numpy().astype(int).tolist())
    assert ids == [e[2] for e in expect]


@pytest.mark.parametrize('case_id', [0, 1, 2])
def test_ssar_staging_matches_reference_wrapper(golden, case_id):
    from surreal_b200.replay import UniformReplay
    from surreal_b200.env import ExpSenderWrapperSSARNStepBootstrap as W
    case = golden('window_ssar').js('cases')[case_id]
    n, gamma, ep_lens = case['n_step'], case['gamma'], case['ep_lens']
    lc, ec, sc = ddpg_configs(D=2, A=1, n_step=n, memory_size=64, start=0)
    lc.algo.gamma = gamma
    R = UniformReplay(lc, ec, sc)
    env = ScriptedEnv([ep_lens])
    w = W(env, lc, sc, replay=R)
    w.reset()
    for _ in range(sum(ep_lens)):
        w.step(torch.full((1, 1), float(env.g[0]), device=DEV))
    exp = case['records']
    assert len(R) == len(exp)
    k = len(exp)
    assert R.r_obs[:k, 0].cpu().numpy().astype(int).tolist() == [e['obs'] for e in exp]
    assert R.r_obs_next[:k, 0].cpu().numpy().astype(int).tolist() == [e['obs_next'] for e in exp]
    assert R.r_act[:k, 0].cpu().numpy().tolist() == [e['action'] for e in exp]
    assert R.r_done[:k].cpu().numpy().astype(bool).tolist() == [e['done'] for e in exp]
    np.testing.assert_array_equal(R.r_rew[:k].cpu().numpy(), np.array([e['reward'] for e in exp], dtype=np.float32))
    # and against the oracle model for a multi-actor run (slot = k-th emission in (step, actor) order)
    got = ssar_nstep(ep_lens, n, gamma, lambda g: 0.25 * g - 3.0)
    assert [(o, on) for o, on, *_ in got] == [(e['obs'], e['obs_next']) for e in exp]


def test_ppo_agent_act_matches_reference(golden):
    from surreal_b200.agent import PPOAgent
    g = golden('ppo_act')
    N = len(g['obs'])
    lc, ec, sc = ppo_configs(D=11, A=3)
    ec.num_envs = N
    ag = PPOAgent(lc, ec, sc, 3, 'training')
    ag.model.load_state_dict(ref_state_dict(g.sub('model/')))
    ag.set_noise(np.full(N, float(g['noise'])))
    action, info = ag.act({'low_dim': {'flat_inputs': g['obs']}}, eps=g['eps'])
    assert action.dtype == np.float64 and action.shape == (N, 3)
    np.testing.assert_allclose(info[1][0], g['pds'], rtol=0, atol=2e-6)
    np.testing.assert_allclose(action, g['actions'], rtol=0, atol=2e-6)
    ag.agent_mode = 'eval_deterministic'
    det = ag.act({'low_dim': {'flat_inputs': g['obs']}})
    np.testing.assert_allclose(det, g['actions_det'], rtol=0, atol=2e-6)


def test_engine_end_to_end_runs_and_is_consistent():
    """replay -> learner -> agent through the launcher; windows the learner consumes are exactly what the
    actors staged (behaviour pd recorded after noise scaling, FIFO order), parameters reach the agent only
    at publish + fetch."""
    from surreal_b200.launch import SurrealDefaultLauncher
    from surreal_b200.agent import PPOAgent
    from surreal_b200.learner import PPOLearner
    from surreal_b200.replay import FIFOReplay
    from surreal_b200.main.ppo_configs import make_synthetic_env_config
    N, n = 64, 8
    lc, ec, sc = ppo_configs(D=16, A=4, actor_h=(64, 48), critic_h=(64, 48), n_step=n, stride=n, B=N,
                             memory_size=2 * N, exp_interval=N)
    make_synthetic_env_config(ec, N, 16, 4, seed=3)
    ec.limit_episode_length = 2 * n
    sc.agent.fetch_parameter_interval = 1
    lc.parameter_publish.min_publish_interval = 0.0        # the reference throttles publishes to one per 0.3 s
    la = SurrealDefaultLauncher(PPOAgent, PPOLearner, FIFOReplay, sc, ec, lc)
    agent, replay, learner = la.setup_engine()
    # like the reference, PPO's first publish only happens after exp_interval experiences (ppo.py:633): until then
    # the actors run their own initial weights
    w0 = agent.model.actor.params.clone()
    assert learner.publisher.version == 0
    agent.main_loop(max_steps=n)
    torch.cuda.synchronize()
    assert len(replay) == N
    pd_first = replay.r_pd[:N, 0].clone()
    expect_std = torch.exp(agent.model.log_var)[None, :] * torch.exp(agent._log_noise)[:, None]
    assert torch.allclose(pd_first[:, 4:], expect_std, rtol=1e-6)
    assert float(replay.r_act[:N].abs().max()) <= 1.0
    learner.main_loop()                                           # consumes the N windows, publishes (exp_interval)
    assert len(replay) == 0 and learner.publisher.version == 1
    assert not torch.equal(learner.model.actor.params, w0)
    assert torch.equal(agent.model.actor.params, w0)              # actors still run the lagged snapshot
    agent.main_loop(max_steps=1)                                  # fetch_parameter_interval = 1 -> pulls the new one
    assert torch.equal(agent.model.actor.params, learner.model.actor.params)
    st = learner.tensorplex.last
    for k in ['_pol_kl', '_val_loss', '_surr_loss', '_entropy', 'grad_norm_actor', 'grad_norm_critic']:
        assert k in st and np.isfinite(st[k])


def test_synthetic_env_dynamics_and_episode_cap():
    """s' = tanh(Ws s + Wa a) + 0.01 xi, r = -|s|^2/D + 0.1 xi', done at the episode cap with auto-reset."""
    from surreal_b200.env import SyntheticEnv
    N, D, A, L = 257, 24, 5, 4
    env = SyntheticEnv(N, D, A, limit_episode_length=L, seed=9)
    obs, _ = env.reset()
    s = obs['low_dim']['flat_inputs'].clone()
    for t in range(1, 2 * L + 1):
        a = torch.rand(N, A, device=DEV) * 2 - 1
        obs2, r, d, info = env.step(a)
        expect = torch.tanh(s @ env.Ws.t() + a @ env.Wa.t())
        assert float((info['obs_next'] - expect).abs().max()) < 0.01 * 6
        assert float((r - (-(s * s).sum(1) / D)).abs().max()) < 0.1 * 6
        is_done = (t % L == 0)
        assert bool((d == (1.0 if is_done else 0.0)).all())
        nxt = obs2['low_dim']['flat_inputs']
        if is_done:
            assert abs(float(nxt.mean())) < 0.1 and abs(float(nxt.std()) - 1.0) < 0.1      # fresh N(0,1) states
            assert bool((env.ep_step == 0).all())
        else:
            assert torch.equal(nxt, info['obs_next'])
        s = nxt.clone()
    noise = (info['obs_next'] - expect)
    assert 0.005 < float(noise.std()) < 0.02


def test_pipelined_engine_matches_sequential_semantics():
    """Two-stream PipelinedEngine: every window is consumed exactly once, in arrival order, and the learner's
    statistics are finite; parameters reach the actors one publish late (the documented policy lag)."""
    from surreal_b200.launch import SurrealDefaultLauncher, PipelinedEngine
    from surreal_b200.agent import PPOAgent
    from surreal_b200.learner import PPOLearner
    from surreal_b200.replay import FIFOReplay
    from surreal_b200.main.ppo_configs import make_synthetic_env_config
    N, n = 128, 8
    lc, ec, sc = ppo_configs(D=16, A=4, actor_h=(64, 48), critic_h=(64, 48), n_step=n, stride=n, B=N,
                             memory_size=2 * N, exp_interval=N)
    make_synthetic_env_config(ec, N, 16, 4, seed=5)
    ec.limit_episode_length = 2 * n
    sc.agent.fetch_parameter_interval = n
    lc.parameter_publish.min_publish_interval = 0.0
    la = SurrealDefaultLauncher(PPOAgent, PPOLearner, FIFOReplay, sc, ec, lc)
    agent, replay, learner = la.setup_engine()
    eng = PipelinedEngine(agent, replay, learner, n)
    eng.prime()
    versions = []
    for k in range(6):
        st = eng.step()
        assert all(np.isfinite(v) for v in st.values())
        versions.append(learner.publisher.version)
    eng.drain()
    s = replay._read_state()
    assert s['total_in'] == 7 * N and s['total_out'] == 6 * N and s['count'] == N and s['dropped'] == 0
    assert versions == [1, 2, 3, 4, 5, 6]
    assert agent._ps_client._last_version in (5, 6)               # one publish behind the learner at most
    assert learner.current_iteration == 6


@pytest.mark.parametrize('n,stride,cap_extra', [(8, 8, 40), (6, 4, 40), (4, 4, -30)])
def test_fused_rollout_launches_match_unfused(n, stride, cap_extra):
    """sample+slot-assignment and env+commit fused launches (3 per step) against the 5-launch sequence: identical
    actions, staging and FIFO contents, including overlapping windows, episode ends and a queue that overflows
    inside ONE step (more completing actors than capacity)."""
    from surreal_b200.agent import PPOAgent
    from surreal_b200.replay import FIFOReplay
    from surreal_b200.env import SyntheticEnv
    N, D, A, T = 50, 12, 3, 37
    out = []
    for fuse in (True, False):
        lc, ec, sc = ppo_configs(D=D, A=A, actor_h=(40, 36), critic_h=(40, 36), n_step=n, stride=stride, B=8,
                                 memory_size=N + cap_extra)
        ec.num_envs = N
        R = FIFOReplay(lc, ec, sc)
        ag = PPOAgent(lc, ec, sc, 1, 'training')
        torch.manual_seed(5)
        ag.model.actor.params.copy_(torch.randn_like(ag.model.actor.params) * 0.2)
        ag.set_noise(np.linspace(-0.5, 0.5, N))                   # the per-actor exploration constant is drawn at random
        env = SyntheticEnv(N, D, A, limit_episode_length=11, seed=4)
        ag.env = w = ag.prepare_env_agent(env)
        w.fuse_launches = fuse
        obs, _ = w.reset()
        acts = []
        for _ in range(T):
            a = ag.act(obs)
            acts.append(a[0].clone())
            obs, _, _, _ = w.step(a)
        torch.cuda.synchronize()
        out.append(dict(acts=torch.stack(acts), state=R._read_state(), pos=w.stage_pos.clone(), so=w.stage_obs.clone(),
                        r_obs=R.r_obs.clone(), r_act=R.r_act.clone(), r_pd=R.r_pd.clone(), r_rew=R.r_rew.clone(),
                        r_done=R.r_done.clone(), ctr=int(env.step_counter.item())))
    f, u = out
    assert f['state'] == u['state'] and f['ctr'] == u['ctr'] == T
    assert f['state']['total_in'] > 0 and (cap_extra > 0 or f['state']['dropped'] > 0)
    for k in ['acts', 'pos', 'r_obs', 'r_act', 'r_pd', 'r_rew', 'r_done']:
        assert torch.equal(f[k], u[k]), k


def _rollout_pair(n, stride, cap_extra, zero_head, T, actor_h=(48, 32), A=3, N=50, D=12):
    """Run the same chunk through the persistent rollout kernel and through the per-step launch sequence."""
    from surreal_b200.agent import PPOAgent
    from surreal_b200.replay import FIFOReplay
    from surreal_b200.env import SyntheticEnv
    out = []
    for persistent in (True, False):
        lc, ec, sc = ppo_configs(D=D, A=A, actor_h=actor_h, critic_h=(48, 32), n_step=n, stride=stride, B=8,
                                 memory_size=N + cap_extra)
        ec.num_envs = N
        R = FIFOReplay(lc, ec, sc)
        ag = PPOAgent(lc, ec, sc, 1, 'training')
        torch.manual_seed(5)
        ag.model.actor.params.copy_(torch.randn_like(ag.model.actor.params) * 0.2)
        if zero_head:                                             # mean == tanh(0) == 0 on both paths: bitwise comparable
            ag.model.actor.W(2).zero_()
            ag.model.actor.b(2).zero_()
        ag.model.z_stats.copy_(torch.cat([torch.linspace(-3, 3, D) * 10, torch.linspace(1, 2, D) * 40,
                                          torch.tensor([10.0])]).to(DEV))
        ag.set_noise(np.linspace(-0.5, 0.5, N))
        env = SyntheticEnv(N, D, A, limit_episode_length=11, seed=4)
        ag.env = w = ag.prepare_env_agent(env)
        obs, _ = w.reset()
        if persistent:
            assert ag.rollout_chunk_supported()
            for t0 in range(0, T, 8):                             # several chunks: state carries over between launches
                assert ag.rollout_chunk(min(8, T - t0))
        else:
            for _ in range(T):
                a = ag.act(obs)
                obs, _, _, _ = w.step(a)
        torch.cuda.synchronize()
        out.append(dict(state=R._read_state(), ctr=int(env.step_counter.item()), pos=w.stage_pos.clone(),
                        ep=env.ep_step.clone(), env_state=env.state.clone(), act=ag._action.clone(), pd=ag._pd.clone(),
                        rew=env.reward.clone(), done=env.done.clone(), obs_next=env.obs_next.clone(),
                        r_obs=R.r_obs.clone(), r_act=R.r_act.clone(), r_pd=R.r_pd.clone(), r_rew=R.r_rew.clone(),
                        r_done=R.r_done.clone(), so=w.stage_obs.clone(), sa=w.stage_act.clone()))
    return out


# 96x64-A32: a policy whose head's k-slice sums need more of the kernel's partial-sum buffer than its hidden layers do
@pytest.mark.parametrize('n,stride,cap_extra,actor_h,A', [
    pytest.param(8, 8, 40, (48, 32), 3, id='8-8-40'), pytest.param(6, 4, 40, (48, 32), 3, id='6-4-40'),
    pytest.param(4, 4, -30, (48, 32), 3, id='4-4--30'), pytest.param(5, 2, 100, (48, 32), 3, id='5-2-100'),
    pytest.param(8, 8, 40, (96, 64), 32, id='8-8-40-96x64-A32')])
def test_persistent_rollout_matches_per_step_bitwise(n, stride, cap_extra, actor_h, A):
    """One persistent launch per chunk vs T x (forward, sample, env+commit): with a zero policy head both paths
    produce mean == 0 exactly, so sampling, env dynamics, window staging (overlapping windows, episode ends),
    outbox -> FIFO ordering in (step, actor) order and drop-oldest must agree bit for bit."""
    p, s = _rollout_pair(n, stride, cap_extra, zero_head=True, T=29, actor_h=actor_h, A=A)
    assert p['state'] == s['state'] and p['ctr'] == s['ctr'] == 29
    assert p['state']['total_in'] > 0 and (cap_extra > 0 or p['state']['dropped'] > 0)
    for k in ['pos', 'ep', 'env_state', 'act', 'pd', 'rew', 'done', 'obs_next', 'r_obs', 'r_act', 'r_pd', 'r_rew',
              'r_done', 'sa']:
        assert torch.equal(p[k], s[k]), k


def test_persistent_rollout_policy_forward_close():
    """Same comparison with a live policy head: the cluster FFMA forward and the per-step tensor-core forward agree
    to fp32 rounding, so trajectories stay within a small tolerance and every discrete quantity is identical.  The
    second policy has a head whose k-slice sums need more of the kernel's partial-sum buffer than its hidden layers do."""
    for actor_h, A in (((48, 32), 3), ((96, 64), 32)):
        p, s = _rollout_pair(8, 8, 40, zero_head=False, T=16, actor_h=actor_h, A=A)
        assert p['state'] == s['state'] and torch.equal(p['pos'], s['pos']) and torch.equal(p['ep'], s['ep'])
        assert torch.equal(p['r_done'], s['r_done'])
        d0 = (p['r_pd'][:, 0, :A] - s['r_pd'][:, 0, :A]).abs().max()           # first step: identical inputs
        assert float(d0) <= 1e-5, (actor_h, float(d0))
        assert float(p['r_pd'][:, 0, :A].abs().max()) > 0.05                       # ... and a non-trivial policy output
        for k in ['r_obs', 'r_act', 'r_pd', 'r_rew', 'env_state']:
            assert float((p[k] - s[k]).abs().max()) <= 2e-3, (actor_h, k, float((p[k] - s[k]).abs().max()))


class NumpyScriptEnv:
    """Batched HOST env (numpy in / numpy out): deterministic observations, rewards and episode ends."""

    def __init__(self, N, D, A, ep_len):
        self.N, self.D, self.A, self.ep_len = N, D, A, ep_len
        self.t = 0
        self.seen_actions = []

    def _obs(self, t):
        i = np.arange(self.N, dtype=np.float32)[:, None]
        d = np.arange(self.D, dtype=np.float32)[None, :]
        return np.sin(0.1 * t + i + 0.01 * d).astype(np.float32)

    def reset(self):
        self.t = 0
        return {'low_dim': {'flat_inputs': self._obs(0)}}, {}

    def step(self, action):
        assert isinstance(action, np.ndarray) and action.shape == (self.N, self.A)
        self.seen_actions.append(action.astype(np.float32))
        self.t += 1
        done = np.full(self.N, float(self.t % self.ep_len == 0), dtype=np.float32)
        rew = (self.t + np.arange(self.N) / 1000.0).astype(np.float32)
        nxt = self._obs(self.t)
        return {'low_dim': {'flat_inputs': nxt}}, rew, done, {'obs_next': nxt}


def test_host_env_actor_loop_stages_windows_in_hbm():
    """agent.act(numpy) -> host env.step(numpy) -> wrapper.step: observations / rewards / dones cross PCIe per step and
    the windows land in the HBM FIFO in (step, actor) order with exactly the host's values; the exploration noise
    advances every step (shared Philox counter owned by the wrapper)."""
    from surreal_b200.agent import PPOAgent
    from surreal_b200.replay import FIFOReplay
    N, D, A, n, T = 6, 8, 3, 4, 16
    lc, ec, sc = ppo_configs(D=D, A=A, actor_h=(32, 16), critic_h=(32, 16), n_step=n, stride=n, B=4, memory_size=64)
    ec.num_envs = N
    R = FIFOReplay(lc, ec, sc)
    ag = PPOAgent(lc, ec, sc, 0, 'training')
    env = NumpyScriptEnv(N, D, A, ep_len=8)
    ag.env = w = ag.prepare_env_agent(env)
    assert w.host_env
    obs, _ = w.reset()
    pds = []
    for _ in range(T):
        a = ag.act(obs)
        assert isinstance(a[0], np.ndarray) and a[0].dtype == np.float64
        pds.append(a[1][1][0].copy())
        obs, _, _, _ = w.step(a)
    torch.cuda.synchronize()
    st = R._read_state()
    assert st['count'] == N * (T // n) and int(w.step_counter.item()) == T
    # the one-call host path (sb200_ppo_act_host_f32) and the generic device-tensor path compute the same policy output
    ag.agent_mode = 'eval_deterministic'
    o = env._obs(3)
    np.testing.assert_array_equal(ag.act(o), ag.act(torch.tensor(o, device=DEV)).cpu().numpy().astype(np.float64))
    ag.agent_mode = 'training'
    acts = np.stack(env.seen_actions)                              # [T, N, A]
    assert np.abs(acts[1] - acts[0]).max() > 1e-3                  # fresh noise every step
    for k in range(T // n):                                        # completion step n*(k+1)-1, actors in order
        for i in range(N):
            b = R.sample(1)
            t0 = k * n
            exp_obs = np.stack([env._obs(t0 + j)[i] for j in range(n)])
            np.testing.assert_array_equal(b['obs']['low_dim']['flat_inputs'][0].cpu().numpy(), exp_obs)
            np.testing.assert_array_equal(b['obs_next']['low_dim']['flat_inputs'][0, 0].cpu().numpy(), env._obs(t0 + n)[i])
            np.testing.assert_array_equal(b['actions'][0].cpu().numpy(), acts[t0:t0 + n, i])
            np.testing.assert_array_equal(b['persistent_infos'][0][0].cpu().numpy(), np.stack([pds[t0 + j][i] for j in range(n)]))
            np.testing.assert_array_equal(b['rewards'][0].cpu().numpy(),
                                          np.array([t0 + j + 1 + i / 1000.0 for j in range(n)], dtype=np.float32))
            np.testing.assert_array_equal(b['dones'][0].cpu().numpy(),
                                          np.array([float((t0 + j + 1) % 8 == 0) for j in range(n)], dtype=np.float32))
