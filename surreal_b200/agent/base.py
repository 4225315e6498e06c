"""Agent base class: constructor, hooks and main loop of surreal/agent/base.py:24-377, for a BATCH of
co-located actors.

One Agent object drives ``num_envs`` actors that share the GPU (the reference runs one OS process per
actor with a batch-1 forward each, launcher.py:181-232).  The parameter wire is the in-process
ParameterClient of ``surreal_b200.distributed``: ``fetch_parameter()`` copies the learner's last PUBLISHED
snapshot into this agent's own model, so between fetches the actors run lagged weights exactly as
Surreal's do (fetch cadence: session_config.agent.fetch_parameter_mode/interval, base.py:182-207)."""
import time

from .. import utils as U
from ..distributed import ParameterClient, ModuleDict, LocalHub

AGENT_MODES = ['training', 'eval_deterministic', 'eval_stochastic', 'eval_deterministic_local',
               'eval_stochastic_local']


class Agent(metaclass=U.AutoInitializeMeta):
    def __init__(self, learner_config, env_config, session_config, agent_id, agent_mode, render=False):
        self.learner_config = learner_config
        self.env_config = env_config
        self.session_config = session_config
        assert agent_mode in AGENT_MODES
        self.agent_mode = agent_mode
        self.agent_id = agent_id
        self.render = render
        self.num_envs = int(env_config.num_envs) if 'num_envs' in env_config else 1
        if self.agent_mode not in ['eval_deterministic_local', 'eval_stochastic_local']:
            self._fetch_parameter_mode = self.session_config.agent.fetch_parameter_mode
            self._fetch_parameter_interval = self.session_config.agent.fetch_parameter_interval
            self._fetch_parameter_tracker = U.PeriodicTracker(self._fetch_parameter_interval)
            self.log = U.get_logger('agent-%s' % agent_id)
            self.tensorplex = U.ScalarSink('agent/%s' % agent_id)
            self.actions_per_param_update = U.MovingAverageRecorder(decay=0.99)
            self.episodes_per_param_update = U.MovingAverageRecorder(decay=0.99)
        self.current_episode = 0
        self.cumulative_steps = 0
        self.current_step = 0
        self.actions_since_param_update = 0
        self.episodes_since_param_update = 0
        self.env = None
        self._rollout_graphs = {}
        self._in_chunk = False                 # True while main_loop() records / runs a multi-step chunk

    def _initialize(self):
        if self.agent_mode not in ['eval_deterministic_local', 'eval_stochastic_local']:
            md = self.module_dict()
            self._module_dict = md if isinstance(md, ModuleDict) else ModuleDict(md)
            self._ps_client = ParameterClient(LocalHub.get(self.session_config).publisher)

    # -- abstract ---------------------------------------------------------------------------------------
    def act(self, obs):
        raise NotImplementedError

    def module_dict(self):
        raise NotImplementedError

    # -- hooks (agent/base.py:160-218) ------------------------------------------------------------------
    def on_parameter_fetched(self, params, info):
        if self.agent_mode == 'training':
            self.actions_per_param_update.add_value(self.actions_since_param_update)
            self.episodes_per_param_update.add_value(self.episodes_since_param_update)
            self.tensorplex.add_scalars({
                '.core/parameter_publish_delay_s': time.time() - info['time'],
                '.core/actions_per_param_update': self.actions_per_param_update.cur_value(),
                '.core/episodes_per_param_update': self.episodes_per_param_update.cur_value()})
            self.actions_since_param_update = 0
            self.episodes_since_param_update = 0
        return params

    def pre_action(self, obs):
        if self.agent_mode == 'training':
            if self._fetch_parameter_mode == 'step' and self._fetch_parameter_tracker.track_increment():
                self.fetch_parameter()

    def post_action(self, obs, action, obs_next, reward, done, info):
        self.current_step += 1
        self.cumulative_steps += self.num_envs
        if self.agent_mode == 'training':
            self.actions_since_param_update += 1

    def pre_episode(self):
        if self.agent_mode == 'training':
            if self._fetch_parameter_mode == 'episode' and self._fetch_parameter_tracker.track_increment():
                self.fetch_parameter()

    def post_episode(self):
        self.current_episode += 1

    # -- main loop (agent/base.py:224-271) --------------------------------------------------------------
    def main(self):
        self.main_setup()
        while True:
            self.main_loop()

    def main_setup(self, env=None):
        env = env if env is not None else self.get_env()
        self.env = self.prepare_env(env)
        if self.agent_mode == 'training':
            self.fetch_parameter()
        self._obs = None

    def main_loop(self, max_steps=None):
        """One 'episode' of the batched env: ``limit_episode_length`` steps of ALL actors (actors whose episode
        ends earlier are auto-reset on the device, their windows never span episodes)."""
        env = self.env
        self.pre_episode()
        if self._obs is None:
            self._obs, _ = env.reset()
        steps = max_steps if max_steps is not None else max(int(self.env_config.limit_episode_length), 1)
        obs = self._obs
        if self._device_resident(obs):
            # device-resident env: the whole chunk is a fixed launch sequence with no host logic inside -- ONE
            # persistent kernel where the policy / env allow it, else act -> env -> staging kernels x steps -- submitted
            # as one CUDA graph (SB200_CUDA_GRAPH=0: the same launches, eagerly).  Parameter fetches happen at chunk
            # boundaries, at the configured cadence.
            from ..ops import GraphRunner, graphs_enabled
            if self.agent_mode == 'training' and self._fetch_parameter_mode == 'step' and \
                    self._fetch_parameter_tracker.track_increment(steps):
                self.fetch_parameter()
            persistent = hasattr(self, 'rollout_chunk') and self.rollout_chunk_supported()
            if persistent:
                env.rollout_outbox(steps)              # allocate outside graph capture

            def body():
                if persistent and self.rollout_chunk(steps):
                    return                             # whole chunk = one persistent kernel + the commit pass
                o = obs
                packed = getattr(self, '_packed', None)
                if packed is not None:
                    packed.refresh()                   # weights are fixed inside a chunk: pack them once, here
                self._in_chunk = True
                try:
                    for _ in range(steps):
                        a = self.act(o)
                        o, _, _, _ = env.step(a)
                finally:
                    self._in_chunk = False
            if graphs_enabled():
                if steps not in self._rollout_graphs:
                    self._rollout_graphs[steps] = GraphRunner()
                self._rollout_graphs[steps].run(body)
            else:
                body()
            self.current_step += steps
            self.cumulative_steps += steps * self.num_envs
            self.actions_since_param_update += steps
            self.post_episode()
            return
        for _ in range(steps):
            self.pre_action(obs)
            action = self.act(obs)
            obs_next, reward, done, info = env.step(action)
            self.post_action(obs, action, obs_next, reward, done, info)
            obs = obs_next
        self._obs = obs
        self.post_episode()

    def _device_resident(self, obs):
        """The chunked path needs every buffer of the step to live at a fixed device address: true for the in-tree
        device env (its obs tensor is its state buffer), false for host envs."""
        if not getattr(self.env, 'graph_safe', False):
            return False
        import torch
        from ..utils import obs_flat
        x = obs_flat(obs)
        return isinstance(x, torch.Tensor) and x.is_cuda

    def get_env(self):
        from ..env import SyntheticEnv
        ec = self.env_config
        name = ec.env_name if 'env_name' in ec else ''
        if not str(name).startswith('synthetic'):
            raise ValueError('only the device-resident synthetic env ships with surreal_b200 (env_name "synthetic"); '
                             'gym / dm_control / robosuite adapters are out of scope -- pass your own env to '
                             'main_setup(env)')
        from ..utils import obs_is_pixel, obs_is_mixed
        if obs_is_mixed(ec.obs_spec):
            from ..env import SyntheticMixedEnv
            return SyntheticMixedEnv(self.num_envs, ec.obs_spec, ec.action_spec.dim[0], ec.limit_episode_length,
                                     seed=int(ec.seed) if 'seed' in ec else 0)
        if obs_is_pixel(ec.obs_spec):
            from ..env import SyntheticPixelEnv
            return SyntheticPixelEnv(self.num_envs, tuple(ec.obs_spec['pixel']['camera0']), ec.action_spec.dim[0],
                                     ec.limit_episode_length, seed=int(ec.seed) if 'seed' in ec else 0)
        D = sum(v[0] for v in ec.obs_spec['low_dim'].values())
        return SyntheticEnv(self.num_envs, D, ec.action_spec.dim[0], ec.limit_episode_length,
                            seed=int(ec.seed) if 'seed' in ec else 0)

    def prepare_env(self, env):
        return self.prepare_env_agent(env) if self.agent_mode == 'training' else self.prepare_env_eval(env)

    def prepare_env_agent(self, env):
        return env

    def prepare_env_eval(self, env):
        return env

    def main_agent(self):
        self.main()

    def main_eval(self):
        self.main()

    # -- parameters -------------------------------------------------------------------------------------
    def fetch_parameter(self):
        if self._ps_client._publisher is None:
            self._ps_client.attach(LocalHub.get(self.session_config).publisher)
        params, info = self._ps_client.fetch_parameter_with_info()
        if params:
            params = self.on_parameter_fetched(params, info)
            self._module_dict.load(params)

    def fetch_parameter_info(self):
        return self._ps_client.fetch_info()

    def set_agent_mode(self, agent_mode):
        assert agent_mode in AGENT_MODES
        self.agent_mode = agent_mode
