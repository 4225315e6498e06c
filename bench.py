#!/usr/bin/env python
"""Benchmark of the hot path on BASELINE.json's headline config.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[1] -- PPO, synthetic 64-dim observations, 1024 actors x
horizon 128 (n_step = stride = 128), 2x256 MLP actor + critic, clip mode, z-filter on, A = 8.
One "step" = one pass of the hot path over one batch: a 128-step rollout of all 1024 co-located actors
(batched policy inference -> device env -> window staging -> HBM FIFO replay) followed by one
PPOLearner.learn() on the 1024 windows (critic pass over 132 096 rows -> windowed GAE -> <=10 clipped-
surrogate policy epochs with KL early stop -> 10 value epochs), then publish + actor fetch.

  value  : env-steps/s of the whole job, data resident in HBM (device actors feeding the device learner).
  e2e    : the same metric through the reference-facing plugin API with HOST buffers: PPOAgent.act(numpy obs)
           per env step (H2D obs, D2H action + pd) and PPOLearner.learn(numpy batch) (H2D batch, D2H stats).
  roofline: the dominant kernel of the step (the fused critic pass), timed live with CUDA events.
  cpu_baseline / --impl reference: the CPU oracle (a line-by-line restatement of the reference's torch-CPU
           actors + learner, pinned against reference-generated goldens) timed on this box's host cores.
Timing: CUDA events on the launching stream, >= 3 warm-up steps, max over ranks; inputs of every step are
freshly generated on the device (the 47 MB batch and ~60 MB of staging/replay traffic per step exceed any
reuse window together with the explicit L2 flush between timed steps).
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ACTORS, HORIZON, OBS_DIM, ACT_DIM, HIDDEN = 1024, 128, 64, 8, (256, 256)
EPISODE_LEN = 256          # two windows per episode (windows never span episodes)


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d['hbm_gbs'], bf16_tflops=d['bf16_tflops'], bf16_tflops_sustained=d.get('bf16_tflops_sustained'),
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source='fallback (B200_PROFILING.md)')


def build_configs(n_actors=N_ACTORS, horizon=HORIZON):
    from surreal_b200.session import Config
    from surreal_b200.main.ppo_configs import (PPO_DEFAULT_LEARNER_CONFIG, PPO_DEFAULT_ENV_CONFIG,
                                               PPO_DEFAULT_SESSION_CONFIG, make_synthetic_env_config)
    lc = Config(copy.deepcopy(PPO_DEFAULT_LEARNER_CONFIG.to_dict()))
    ec = Config(copy.deepcopy(PPO_DEFAULT_ENV_CONFIG.to_dict()))
    sc = Config(copy.deepcopy(PPO_DEFAULT_SESSION_CONFIG.to_dict()))
    sc.folder = tempfile.mkdtemp(prefix='sb200_bench_')
    lc.model.actor_fc_hidden_sizes = list(HIDDEN)
    lc.model.critic_fc_hidden_sizes = list(HIDDEN)
    lc.algo.ppo_mode = 'clip'
    lc.algo.rnn.if_rnn_policy = False
    lc.algo.n_step = horizon
    lc.algo.stride = horizon
    lc.replay.batch_size = n_actors
    lc.replay.memory_size = 2 * n_actors
    lc.parameter_publish.exp_interval = n_actors          # publish after every learn()
    lc.parameter_publish.min_publish_interval = 0.0
    make_synthetic_env_config(ec, n_actors, OBS_DIM, ACT_DIM, seed=0)
    ec.limit_episode_length = EPISODE_LEN
    sc.agent.fetch_parameter_interval = horizon
    return lc, ec, sc


def load_profile_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, as recorded in profiles/traffic.json from the
    committed `ncu --set full` captures (tools/summarize_profiles.py writes it); None when no capture is on file."""
    p = os.path.join(ROOT, 'profiles', 'traffic.json')
    try:
        return json.load(open(p)).get(kernel, {}).get('dram_bytes')
    except Exception:                                             # noqa: BLE001
        return None


WORKLOAD = 'cfg2'          # --workload cfg5: BASELINE configs[4], 4096 actors x horizon 256 in TOTAL (strong scaling)


def bench_config(world):
    """The `config` object of BOTH arms' JSON lines (identical: same workload, same keys, same values)."""
    if WORKLOAD == 'cfg5':
        return {'workload': 'PPO synthetic 64-dim obs, 4096 actors x horizon 256 in total, 2x256 MLP, data-parallel learner '
                            '(BASELINE configs[4])',
                'actors_per_gpu': N_ACTORS, 'horizon': HORIZON, 'obs_dim': OBS_DIM, 'action_dim': ACT_DIM, 'hidden': list(HIDDEN),
                'ppo_mode': 'clip', 'epoch_policy': 10, 'epoch_baseline': 10, 'episode_length': EPISODE_LEN,
                'global_windows_per_step': N_ACTORS * world, 'parallelism': 'dp%d' % world,
                'l2': 'flushed between timed steps (192 MB fill)'}
    return {'workload': 'PPO synthetic 64-dim obs, 1024 actors x horizon 128, 2x256 MLP (BASELINE configs[1])',
            'actors_per_gpu': N_ACTORS, 'horizon': HORIZON, 'obs_dim': OBS_DIM, 'action_dim': ACT_DIM, 'hidden': list(HIDDEN),
            'ppo_mode': 'clip', 'epoch_policy': 10, 'epoch_baseline': 10, 'episode_length': EPISODE_LEN,
            'global_windows_per_step': N_ACTORS * world, 'parallelism': 'dp%d' % world,
            'l2': 'flushed between timed steps (192 MB fill)'}


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region.  The timed region is tens of milliseconds, far shorter
    than nvidia-smi's start-up, so the samples come from NVML directly (pynvml, 2 ms polling thread)."""

    def __init__(self, index=0):
        self.index, self.rows, self._run, self._thr, self.h, self.err = index, [], False, None, None, None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            # LOCAL_RANK indexes CUDA_VISIBLE_DEVICES; NVML enumerates physical devices
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(vis.split(',')[index]) if vis and all(v.strip().isdigit() for v in vis.split(',')) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:                                    # noqa: BLE001
            self.err = repr(e)

    def _poll(self):
        nv = self.nv
        while self._run:
            try:
                self.rows.append((int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)),
                                  int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))))
            except Exception as e:                                # noqa: BLE001
                self.err = repr(e)
                return
            time.sleep(0.002)

    def start(self):
        if self.h is None:
            return
        self._run = True
        self._thr = threading.Thread(target=self._poll, daemon=True)
        self._thr.start()

    def stop(self):
        if self.h is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['NVML unavailable: %s' % self.err]}
        self._run = False
        self._thr.join(timeout=1.0)
        nv = self.nv
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for r in self.rows:
            bits |= r[1]
        names = [('hw_slowdown', nv.nvmlClocksEventReasonHwSlowdown), ('hw_thermal_slowdown', nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ('sw_thermal_slowdown', nv.nvmlClocksEventReasonSwThermalSlowdown), ('sw_power_cap', nv.nvmlClocksEventReasonSwPowerCap)]
        reasons = [n for n, b in names if bits & b]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': self.max_mhz, 'reasons': reasons, 'samples': len(sm),
                'source': 'NVML polled every 2 ms during the timed region'}


# --------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        # small messages (600 KB gradients, scalars): a few channels are plenty, and a collective kernel must always
        # find free SMs next to the persistent rollout kernel (128 of 148 SMs) and the other branch's collective
        os.environ.setdefault('NCCL_MAX_NCHANNELS', '4')
        dist.init_process_group('nccl', device_id=dev)
    import __graft_entry__
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()
    from surreal_b200 import _lib
    from surreal_b200.launch import SurrealDefaultLauncher
    from surreal_b200.agent import PPOAgent
    from surreal_b200.learner import PPOLearner
    from surreal_b200.replay import FIFOReplay
    from surreal_b200.distributed import LocalHub
    _lib.lib()
    import numpy as np
    lc, ec, sc = build_configs(N_ACTORS, HORIZON)
    ec.seed = rank
    torch.manual_seed(0)                                          # initial actor / critic weights
    la = SurrealDefaultLauncher(PPOAgent, PPOLearner, FIFOReplay, sc, ec, lc)
    agent, replay, learner = la.setup_engine()
    # the launcher draws the actors' exploration scales from a clock-seeded generator (as the reference does); fix them
    # so that every run with the same arguments sees the same inputs
    agent.set_noise(np.random.default_rng(rank).uniform(-agent.log_sig_range, agent.log_sig_range, agent.num_envs))
    if world > 1:
        learner.enable_data_parallel(dist.group.WORLD)
    N, T, D, A = N_ACTORS, HORIZON, OBS_DIM, ACT_DIM
    flush = torch.empty(192 * 1024 * 1024 // 4, device=dev)       # > 126 MB L2
    launches = {'n': 0}

    from surreal_b200.launch import PipelinedEngine
    eng = None
    if not args.sequential:
        # actors and learner on two concurrent CUDA streams (Surreal's async actor / learner processes on one GPU)
        eng = PipelinedEngine(agent, replay, learner, T)
        eng.prime()

    def seq_step():
        agent.main_loop(max_steps=T)
        learner.main_loop()

    one_step = eng.step if eng is not None else seq_step
    tstream = eng.sL if eng is not None else torch.cuda.current_stream()

    # kernel-launch accounting (ours only): launches per step are counted once via the library's own counter
    for _ in range(max(args.warmup, 3)):
        one_step()
    torch.cuda.synchronize()
    per_step_launches = count_launches(one_step)
    torch.cuda.synchronize()

    clocks = ClockSampler(local)
    times = []
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks.start()
    t_wall0 = time.time()
    for _ in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(tstream):
            flush.fill_(1.0)                                      # L2 flush between timed iterations
            e0.record()
        one_step()
        with torch.cuda.stream(tstream):
            e1.record()
        times.append((e0, e1))
    torch.cuda.synchronize()
    t_wall = time.time() - t_wall0
    clk = clocks.stop()
    ms = [a.elapsed_time(b) for a, b in times]
    total_ms = sum(ms)
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    env_steps = N * T * args.steps * world
    value = env_steps / (total_ms / 1e3)
    opt_steps = sum(learner.epoch_history[-args.steps:]) if hasattr(learner, 'epoch_history') else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, replay, learner)
    # the two halves of a step in isolation (graph-replayed, sequential, device-timed): explains the pipelined number
    phase = {'rollout': [], 'learn': []}
    for _ in range(5):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        agent.main_loop(max_steps=T)
        ev[1].record()
        learner.main_loop()
        ev[2].record()
        torch.cuda.synchronize()
        phase['rollout'].append(ev[0].elapsed_time(ev[1]))
        phase['learn'].append(ev[1].elapsed_time(ev[2]))
    phase_ms = {k: sorted(v)[len(v) // 2] for k, v in phase.items()}
    # roofline of the dominant kernel (fused critic pass) and of the GAE kernel: separate, untimed-for-throughput
    # pass that runs learn() EAGERLY with CUDA events around those two launches (events cannot sit inside a graph)
    _lib.profile_calls(True)
    learner.profile_events = True                                 # -> eager learn(), same launch sequence
    os.environ['SB200_CUDA_GRAPH'] = '0'                          # -> eager rollout
    n_prof = 3
    for _ in range(n_prof):
        flush.fill_(1.0)
        seq_step()                                                # sequential + eager: one CUDA-event pair per call
    os.environ['SB200_CUDA_GRAPH'] = '1'
    learner.profile_events = False
    calls = _lib.profile_calls(False)
    crit_ms = learner.pop_profile('critic_pass')
    learner.pop_profile('gae')
    per_step = {k: (c / n_prof, ms / n_prof, ms / c) for k, (c, ms) in calls.items()}
    total_kernel_ms = sum(v[1] for v in per_step.values())
    breakdown = [{'call': k, 'launches_per_step': round(v[0], 1), 'ms_per_step': round(v[1], 4), 'avg_us': round(v[2] * 1e3, 2),
                  'share': round(v[1] / total_kernel_ms, 4)}
                 for k, v in sorted(per_step.items(), key=lambda kv: -kv[1][1])]
    peaks = load_peaks()
    rows = N * (T + 1)
    w_params = D * HIDDEN[0] + HIDDEN[0] * HIDDEN[1]

    def mlp_roof(key, nrows, out_dim, kernel):
        if key not in per_step:
            return None
        avg_ms = per_step[key][2]
        flop = 2.0 * nrows * (w_params + HIDDEN[1] * out_dim)
        byts = nrows * (D * 4 + out_dim * 4) + (w_params + HIDDEN[1] * out_dim) * 4
        ach = flop / (avg_ms / 1e3) / 1e12
        return {'kernel': kernel, 'bound': 'tensor', 'achieved': ach, 'peak': peaks['bf16_tflops'], 'unit': 'TFLOP/s',
                'frac': ach / peaks['bf16_tflops'], 'traffic': None, 'avg_ms': avg_ms, 'launches_per_step': per_step[key][0],
                'share_of_step_kernel_time': per_step[key][1] / total_kernel_ms, 'algorithmic_flop': flop,
                'algorithmic_bytes': byts, 'achieved_gbs': byts / (avg_ms / 1e3) / 1e9, 'peak_source': peaks['source'],
                'note': 'fp32-accurate 3xTF32 tensor-core path (the 1e-5 parity bar rules out plain TF32/bf16: every '
                        'product costs 3 mma); dense-bf16 tensor peak is the mandated denominator.  At %d rows the '
                        'kernel is a chain of dependent latencies, not a throughput problem' % nrows}
    roof_small = mlp_roof('sb200_mlp_forward_packed_f32[rows=%d]' % N, N, A,
                          'mlp_fwd_pk_kernel (per-env-step policy forward of %d actors, 2-CTA clusters)' % N)
    roof_mb = mlp_roof('sb200_mlp_forward_f32[rows=%d]' % N, N, A,
                       'mlp_fwd_mma_kernel<1> (learner minibatch forward on %d rows)' % N)
    roof_critic = None
    if 'sb200_mlp_forward_tc5_f32' in per_step:
        roof_critic = mlp_roof('sb200_mlp_forward_tc5_f32', rows, 1,
                               'tc5_prep_kernel + mlp3_tc5_kernel (fused critic pass over %d rows: tcgen05.mma kind::tf32 tiles of '
                               '128 rows, accumulators in TMEM, weight images streamed by the TMA engine, 3xTF32)' % rows)
        roof_critic['note'] = ('fp32-accurate 3xTF32: every algorithmic product is 3 tensor-core MMAs, so the tensor pipe executes 3x '
                               'the algorithmic FLOP counted here; denominator = measured dense bf16 peak (the mandated one), the '
                               'tf32 pipe peaks at half of it')
        roof_critic['tensor_pipe_tflops_executed'] = 3.0 * roof_critic['achieved']
    else:
        roof_critic = mlp_roof('sb200_mlp_forward_f32[rows=%d]' % rows, rows, 1,
                               'mlp_fwd_mma_kernel<2> (fused critic pass over %d rows, 3xTF32 mma.sync, 2 CTAs/SM)' % rows)
    roof_roll = None
    rk = 'sb200_ppo_rollout_f32'
    if rk in per_step:
        avg_ms = per_step[rk][2]
        flop = 2.0 * N * T * (w_params + HIDDEN[1] * A + D * (D + A))          # policy forward + env step, all T steps
        byts = N * T * (D + 3 * A + 2) * 4 + 2 * N * ((T + 1) * D + 3 * T * A + 2 * T) * 4   # staging writes + window copy
        ach = flop / (avg_ms / 1e3) / 1e12
        ffma_peak = 148 * 128 * 2 * 1.9e9 / 1e12
        roof_roll = {'kernel': 'ppo_rollout2_kernel (persistent: %d env steps of %d actors per launch; 4-CTA clusters, '
                               'resident weights, warp-specialised env warps, st.async / mbarrier DSMEM hand-offs)' % (T, N),
                     'bound': 'tensor', 'achieved': ach, 'peak': peaks['bf16_tflops'], 'unit': 'TFLOP/s',
                     'frac': ach / peaks['bf16_tflops'], 'traffic': None, 'avg_ms': avg_ms,
                     'launches_per_step': per_step[rk][0], 'share_of_step_kernel_time': per_step[rk][1] / total_kernel_ms,
                     'algorithmic_flop': flop, 'algorithmic_bytes': byts, 'achieved_gbs': byts / (avg_ms / 1e3) / 1e9,
                     'fp32_ffma_peak_tflops': ffma_peak, 'frac_of_fp32_ffma_peak': ach / ffma_peak,
                     'peak_source': peaks['source'],
                     'note': 'fp32 FFMA by necessity (1e-5 parity with the fp32 reference); the dense-bf16 tensor peak is '
                             'the mandated denominator, the fp32 FFMA ceiling (148 SMs x 128 lanes x 2 x 1.9 GHz) the '
                             'meaningful one (tools/fma_bench.cu measures 127 FMA/clk/SM for FFMA and FFMA2 alike).  Per '
                             'step the kernel is a dependent chain: layer -> hand-off -> layer -> hand-off -> '
                             'head / sample / env -> hand-off (profiles/r02b_rollout_trace_*.txt)'}
    # dram__bytes_read.sum + dram__bytes_write.sum per launch, from one `ncu --set full` capture each (profiles/)
    if roof_roll is not None:
        roof_roll['traffic'] = load_profile_traffic('rollout')
    if roof_critic is not None:
        roof_critic['traffic'] = load_profile_traffic('critic')   # dram__bytes of one `ncu --set full` capture (profiles/)
    cands = [r for r in (roof_roll, roof_small, roof_mb, roof_critic) if r is not None]
    roofline = max(cands, key=lambda r: r['share_of_step_kernel_time']) if cands else None
    gae_key = 'sb200_gae_window_f32'
    gae_avg = per_step[gae_key][2] if gae_key in per_step else None
    gae_bytes = N * ((3 * T + 1) * 4 + 8)
    roofline_gae = {'kernel': 'gae_full_kernel', 'bound': 'hbm', 'achieved': gae_bytes / (gae_avg / 1e3) / 1e9 if gae_avg else None,
                    'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'avg_ms': gae_avg, 'algorithmic_bytes': gae_bytes,
                    'frac': (gae_bytes / (gae_avg / 1e3) / 1e9 / peaks['hbm_gbs']) if gae_avg else None,
                    'note': '1.58 MB per launch: below launch latency, cannot approach the HBM roofline stand-alone'}

    e2e = None
    cpu_baseline = None
    extras = None
    if not args.lite:
        # every rank drives its own actors / learner shard through the host API (the learner's collectives need all
        # ranks); the job-level number is all ranks' env-steps over the slowest rank's time
        e2e = run_e2e(agent, learner, lc, dev, steps=max(2, min(args.steps, 5)))
        if world > 1:
            t = torch.tensor([e2e['ms_per_step']], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e['ms_per_step'] = float(t.item())
            e2e['value'] = N * T * world / (e2e['ms_per_step'] / 1e3)
            e2e['h2d_bytes_per_step'] *= world
            e2e['d2h_bytes_per_step'] *= world
        if world == 1 and rank == 0:
            extras = run_extras(dev, peaks, flush)
            cpu_baseline = cpu_reference(steps=3, warmup=1)
    dp_parity = None
    if world > 1:
        dp_parity = dp_parity_check(learner, dev, rank, world)
        dist.barrier()
    if rank == 0:
        out = {
            'metric': 'env-steps/sec', 'value': value, 'unit': 'env-steps/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': max(args.warmup, 3), 'ms_per_step': total_ms / args.steps, 'higher_is_better': True,
            'scaling': 'strong' if WORKLOAD == 'cfg5' else 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': bench_config(world),
            'engine': 'sequential' if eng is None else 'pipelined: actors (stream A) overlap the learner (stream L), '
                      'one-iteration policy lag',
            'learner_updates_per_sec': args.steps / (total_ms / 1e3),
            'optimizer_steps_per_sec': (opt_steps * world / (total_ms / 1e3)) if opt_steps else None,
            'gpu_launches': per_step_launches * args.steps, 'gpu_launches_per_step': per_step_launches,
            'clocks': clk, 'roofline': roofline, 'roofline_critic_pass': roof_critic, 'roofline_gae': roofline_gae,
            'phase_ms_sequential': phase_ms, 'roofline_rollout': roof_roll, 'kernel_breakdown': breakdown[:12], 'e2e': e2e,
            'cpu_baseline': cpu_baseline, 'dp_parity': dp_parity, 'extras': extras, 'wall_s': t_wall, 'wall_env_steps_per_s': env_steps / t_wall / world * world,
        }
        print(json.dumps(out))
    if world > 1:
        # NCCL collectives captured in CUDA graphs make ProcessGroupNCCL's teardown hang (observed on the 2-GPU box:
        # results printed, then the process never exits).  Nothing is left to flush but stdout: leave without
        # running the destructors.
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


DUMP_WINDOWS = 128        # windows per batch-shaped array written by --dump-outputs (a fixed, seeded sample)


def dump_outputs(out_dir, replay, learner):
    """What the last timed step computed, as ``out_dir/<name>.npy`` (float64 statistics, float32 arrays; 12 MB at cfg2, 24 at cfg5):
      stats_*   : the statistics learn() returned;
      *_params  : the learner's parameters after the step (the actor vector ends with log_var), z_stats its z-filter;
      batch_*   : the windows learn() consumed, with the advantages and returns it computed for them;
      replay_*  : the windows the actors left in the replay for the next learn() (none in --sequential mode).
    Batch-shaped arrays hold the same fixed sample of DUMP_WINDOWS window indices."""
    import numpy as np
    import torch
    torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    out = {'stats_' + k.lstrip('_'): np.float64(v) for k, v in learner.tensorplex.last.items()}
    m = learner.model
    out.update(actor_params=m.actor.params, critic_params=m.critic.params, z_stats=m.z_stats)
    B = learner.batch_size
    pick = np.sort(np.random.default_rng(0).choice(B, min(B, DUMP_WINDOWS), replace=False))
    rows = torch.as_tensor(pick, device=learner.device)
    for k, t in learner.replay_out_buffers().items():
        out['batch_' + k] = t[rows]
    out['batch_advantages'], out['batch_returns'] = learner._adv[rows], learner._ret[rows]
    st = replay._read_state()
    if st['count']:
        slots = (st['head'] + rows[rows < st['count']]) % st['capacity']
        for k, t in (('obs_full', replay.r_obs), ('actions', replay.r_act), ('pd', replay.r_pd),
                     ('rewards', replay.r_rew), ('dones', replay.r_done)):
            out['replay_' + k] = t[slots]
    for k, v in out.items():
        if v is None:
            continue
        if isinstance(v, torch.Tensor):
            v = v.detach().float().cpu().numpy()
        np.save(os.path.join(out_dir, k + '.npy'), v)


def run_extras(dev, peaks, flush):
    """Measurements the metric names beside the headline number (bounded: a few seconds):
      gae_sweep : the windowed-GAE kernel at cfg2 (1024 x 128), cfg5 (4096 x 256) and 262 144 windows x 128 -- achieved
                  HBM GB/s on the ALGORITHMIC bytes ((3n+1)*4 read + 8 written per window) vs the measured copy peak;
      ddpg_cfg3 : BASELINE configs[2] -- 1 M-slot UniformReplay in HBM, batch 4096, nets 300-200 / 400-300: replay.sample
                  (CPython-exact host index stream + one fused gather launch), learn() (one CUDA graph), the loop, and
                  the gather kernel alone on a 1 M-sample batch (HBM-bound regime)."""
    import random
    import torch
    from surreal_b200 import ops
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from helpers import ddpg_configs
    from surreal_b200.replay import UniformReplay
    from surreal_b200.replay.base import gather_fields
    from surreal_b200.learner import DDPGLearner
    out = {}

    def dev_time(fn, iters, do_flush=True):
        ms = []
        for _ in range(iters + 2):
            if do_flush:
                flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        ms = sorted(ms[2:])
        return ms[len(ms) // 2]
    sweep = []
    for (B, n, tag) in ((1024, 128, 'cfg2'), (4096, 256, 'cfg5'), (262144, 128, '2^18 windows')):
        g = torch.Generator(device=dev).manual_seed(B)
        r = torch.randn(B, n, device=dev, generator=g)
        v = torch.randn(B, n + 1, device=dev, generator=g)
        d = (torch.rand(B, n, device=dev, generator=g) < 0.01).float()
        adv, ret = torch.empty(B, 1, device=dev), torch.empty(B, 1, device=dev)
        ms = dev_time(lambda: ops.gae_window(r, v, d, 0.995, 0.97, adv=adv, ret=ret), 10)
        byts = B * ((3 * n + 1) * 4 + 8)
        sweep.append({'case': tag, 'windows': B, 'n_step': n, 'ms': ms, 'algorithmic_bytes': byts, 'achieved_gbs': byts / (ms / 1e3) / 1e9,
                      'frac_of_hbm_peak': byts / (ms / 1e3) / 1e9 / peaks['hbm_gbs'], 'launches': 1 if B <= 16384 else 2})
        del r, v, d
    out['gae_sweep'] = {'kernel': 'gae_full_kernel (+ gae_normalize_kernel above 16 384 windows)', 'bound': 'hbm', 'peak': peaks['hbm_gbs'],
                        'unit': 'GB/s', 'cases': sweep, 'l2': 'flushed before every timed launch'}
    D, A, B, CAP = 64, 8, 4096, 1 << 20
    lc, ec, sc = ddpg_configs(D=D, A=A, actor_h=(300, 200), critic_h=(400, 300), B=B, n_step=3, memory_size=CAP, start=3000)
    R = UniformReplay(lc, ec, sc)
    g = torch.Generator(device=dev).manual_seed(4)
    R.r_obs.copy_(torch.randn(CAP, D, device=dev, generator=g))
    R.r_obs_next.copy_(torch.randn(CAP, D, device=dev, generator=g))
    R.r_act.copy_(torch.rand(CAP, A, device=dev, generator=g) * 2 - 1)
    R.r_rew.copy_(torch.randn(CAP, device=dev, generator=g))
    R.r_done.copy_((torch.rand(CAP, device=dev, generator=g) < 0.005).float())
    R.state[0], R.state[1] = 0, CAP
    R.mark_device_inserts()
    L = DDPGLearner(lc, ec, sc)
    random.seed(5)
    for _ in range(5):
        L.learn(R.sample(B))
    torch.cuda.synchronize()
    batch = R.sample(B)
    learn_ms = dev_time(lambda: L.learn(batch), 20, do_flush=False)

    def wall(fn, n):
        torch.cuda.synchronize()
        t0 = time.time()
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
        return (time.time() - t0) * 1e3 / n
    sample_ms = wall(lambda: R.sample(B), 50)
    loop_ms = wall(lambda: L.learn(R.sample(B)), 50)
    rec = (2 * D + A + 2) * 4
    big = 1 << 20
    idx = torch.randint(0, CAP, (big,), device=dev, dtype=torch.int64)
    o = dict(obs=torch.empty(big, D, device=dev), obs_next=torch.empty(big, D, device=dev), act=torch.empty(big, A, device=dev),
             rew=torch.empty(big, 1, device=dev), done=torch.empty(big, 1, device=dev))
    pairs = [(R.r_obs, o['obs'], D), (R.r_obs_next, o['obs_next'], D), (R.r_act, o['act'], A), (R.r_rew, o['rew'], 1), (R.r_done, o['done'], 1)]
    big_ms = dev_time(lambda: gather_fields(pairs, None, idx, big), 10)
    small_ms = dev_time(lambda: gather_fields(pairs, None, idx[:B], B), 10)
    out['ddpg_cfg3'] = {'workload': 'DDPG synthetic 64-dim obs, 1M-slot UniformReplay in HBM, batch 4096, nets 300-200 / 400-300, n_step 3 '
                                    '(BASELINE configs[2])',
                        'learn_ms_device': learn_ms, 'sample_ms_wall': sample_ms, 'loop_ms_wall': loop_ms,
                        'learner_updates_per_sec': 1e3 / loop_ms,
                        'gather': {'kernel': 'gather_multi_kernel (all five record fields, one launch)', 'bound': 'hbm',
                                   'bytes_per_sample': 2 * rec + 8, 'batch_4096_ms': small_ms,
                                   'batch_4096_gbs': B * (2 * rec + 8) / (small_ms / 1e3) / 1e9,
                                   'batch_1M_ms': big_ms, 'batch_1M_gbs': big * (2 * rec + 8) / (big_ms / 1e3) / 1e9,
                                   'batch_1M_frac_of_hbm_peak': big * (2 * rec + 8) / (big_ms / 1e3) / 1e9 / peaks['hbm_gbs'],
                                   'peak': peaks['hbm_gbs'], 'unit': 'GB/s'}}
    return out


def dp_parity_check(learner, dev, rank, world):
    """Correctness evidence a multi-GPU bench line carries with it (the 1-GPU test box cannot run tests/test_dp_gpu.py):
    (1) replica drift of the benchmarked learner after all its steps -- every rank's actor / critic / z-filter state
    must be BIT-identical to rank 0's; (2) one small data-parallel learn() (each rank feeds 1/world of a 256-window
    global batch) against the CPU oracle on the full batch (tests/dp_check.py; the oracle is the checker here)."""
    import torch
    import torch.distributed as dist
    drift = 0.0
    for t in (learner.model.actor.params, learner.model.critic.params, learner.model.z_stats,
              learner.actor_optim.exp_avg, learner.critic_optim.exp_avg_sq):
        if t is None:
            continue
        ref = t.clone()
        dist.broadcast(ref, 0)
        drift = max(drift, float((ref - t).abs().max().item()))
    d = torch.tensor([drift], device=dev, dtype=torch.float64)
    dist.all_reduce(d, op=dist.ReduceOp.MAX)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from dp_check import run_check
    ok, msgs = run_check('clip', False)
    flag = torch.tensor([0.0 if ok else 1.0], device=dev, dtype=torch.float64)
    dist.all_reduce(flag, op=dist.ReduceOp.MAX)
    return {'replica_drift_max_abs': float(d.item()), 'learn_vs_oracle_ok': bool(flag.item() == 0.0),
            'ok': bool(flag.item() == 0.0 and d.item() == 0.0), 'messages_rank0': msgs,
            'check': 'bitwise replica agreement of the benchmarked learner (params, z-filter, Adam moments) + one DP learn() on '
                     'a 256 x 16 global batch vs the CPU oracle on the full batch (advantages, losses, KL <= 1e-5; parameters '
                     'within 2 % of an Adam step; z-filter sums)'}


def count_launches(fn):
    """Count kernel launches of one step with the CUDA profiler-free trick: torch's stream launch counter is not
    exposed, so the library wrappers count their own launches (each C-ABI call = fixed #kernels)."""
    from surreal_b200 import _lib
    _lib.reset_call_counter()
    fn()
    return _lib.call_counter_kernels()


class HostEnv:
    """Batched HOST environment of the e2e measurement: numpy in, numpy out, like a vector of gym envs on the CPU.  The
    dynamics are pre-generated (pinned) so that the host side costs what a real env's output buffer costs -- a
    pointer -- and the number isolates OUR side of the boundary: every observation / reward / done crosses PCIe
    host->device and every action crosses back, each env step."""

    def __init__(self, N, D, A, T, seed=0):
        import numpy as np
        import torch
        self.N, self.D, self.A, self.T = N, D, A, T
        rng = np.random.default_rng(seed)
        self._obs = torch.empty(T + 1, N, D, dtype=torch.float32, pin_memory=True)
        self._obs.numpy()[...] = rng.standard_normal((T + 1, N, D)).astype(np.float32)
        self._rew = torch.empty(T, N, dtype=torch.float32, pin_memory=True)
        self._rew.numpy()[...] = rng.standard_normal((T, N)).astype(np.float32)
        self._done = torch.zeros(T, N, dtype=torch.float32).pin_memory()
        self._done[T - 1] = 1.0                                   # episodes of T steps
        self._o = [self._obs[t].numpy() for t in range(T + 1)]
        self._r = [self._rew[t].numpy() for t in range(T)]
        self._d = [self._done[t].numpy() for t in range(T)]
        self.t = 0

    def reset(self):
        self.t = 0
        return {'low_dim': {'flat_inputs': self._o[0]}}, {}

    def step(self, action):
        assert action.shape == (self.N, self.A)
        t = self.t
        self.t = (t + 1) % self.T
        nxt = self._o[t + 1]
        # the successor is also what the actors observe next (the synthetic stream has no reset transient)
        return {'low_dim': {'flat_inputs': nxt}}, self._r[t], self._d[t], {'obs_next': nxt}


def run_e2e(agent, learner, lc, dev, steps):
    """env-steps/s through the public actor loop with a HOST env: PPOAgent.act(numpy obs) -> env.step(numpy action)
    -> ExpSender wrapper (H2D of obs / reward / done, window staging into the HBM FIFO) x T, then
    learner.main_loop() (sample from the FIFO, learn, publish).  Every env step's inputs cross PCIe host->device
    and its actions device->host inside the timed region; the learner's statistics are read back every step."""
    import torch
    N, T, D, A = N_ACTORS, HORIZON, OBS_DIM, ACT_DIM
    saved_env, saved_obs = agent.env, agent._obs
    henv = HostEnv(N, D, A, T)
    agent.env = w = agent.prepare_env_agent(henv)
    replay = w.replay
    while len(replay) > 0:                                        # start from an empty queue
        replay.sample(min(len(replay), learner.batch_size))

    def step():
        obs, _ = w.reset()
        for _ in range(T):
            a = agent.act(obs)                                    # H2D obs (first step), kernels, D2H action + pd
            obs, _, _, _ = w.step(a)                              # host env; H2D next obs / reward / done; staging
        learner.main_loop()                                       # FIFO -> learn -> publish; D2H statistics

    step()
    torch.cuda.synchronize()
    t0 = time.time()
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    dt = time.time() - t0
    agent.env, agent._obs = saved_env, saved_obs
    h2d = (T + 1) * N * D * 4 + T * 2 * N * 4
    d2h = T * N * (A + 2 * A) * 4 + 32 * 4 + (2 * D + 1) * 4
    return {'value': N * T * steps / dt, 'unit': 'env-steps/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
            'ms_per_step': dt / steps * 1e3, 'steps': steps,
            'api': 'PPOAgent.act(numpy obs) -> HostEnv.step(numpy action) -> ExpSenderWrapper.step x128, then '
                   'PPOLearner.main_loop(); pinned host memory; all copies inside the timed region'}


# --------------------------------------------------------------------------------------------------
# The reference's CPU path, run for real: persistent actor processes + in-process FIFO + torch-CPU learner.
def _ref_layers(dims, gen):
    import torch
    return [((torch.rand(dims[i + 1], dims[i], generator=gen) - 0.5) * 0.2, torch.zeros(dims[i + 1])) for i in range(len(dims) - 1)]


def _ref_actor_proc(rank, nproc, conn, shm_names, n_actors, horizon):
    """One reference actor PROCESS (surreal/agent/base.py:224-271 main loop).  It owns the logical actors
    [rank::nproc] and, per 'go', advances each of them `horizon` env steps exactly as the reference does: batch-1 torch
    forward + numpy Gaussian sampling (ppo_agent.py:106-154), numpy env step, deque windowing with clear-on-done
    (exp_sender_wrapper.py:204-228).  Finished windows are written into shared memory (stands in for the ZeroMQ /
    pyarrow hop, which is omitted); parameters are re-read from shared memory at every 'go' (fetch_parameter)."""
    import numpy as np
    import torch
    from collections import deque
    from multiprocessing import shared_memory
    from oracle.agent import ppo_act
    from oracle.filters import ZFilter
    torch.set_num_threads(1)
    D, A, n = OBS_DIM, ACT_DIM, horizon
    shms = {k: shared_memory.SharedMemory(name=v) for k, v in shm_names.items()}
    dims = [D] + list(HIDDEN) + [A]
    n_par = sum(dims[i] * dims[i + 1] + dims[i + 1] for i in range(3)) + A + 2 * D + 1
    par = np.ndarray((n_par,), dtype=np.float32, buffer=shms['params'].buf)
    w_obs = np.ndarray((n_actors, n, D), dtype=np.float32, buffer=shms['obs'].buf)
    w_next = np.ndarray((n_actors, 1, D), dtype=np.float32, buffer=shms['obs_next'].buf)
    w_act = np.ndarray((n_actors, n, A), dtype=np.float64, buffer=shms['actions'].buf)
    w_rew = np.ndarray((n_actors, n), dtype=np.float64, buffer=shms['rewards'].buf)
    w_done = np.ndarray((n_actors, n), dtype=np.float32, buffer=shms['dones'].buf)
    w_pd = np.ndarray((n_actors, n, 2 * A), dtype=np.float32, buffer=shms['pd'].buf)
    rng = np.random.default_rng(1000 + rank)
    env_rng = np.random.default_rng(0)
    Ws = env_rng.standard_normal((D, D)) / np.sqrt(D)
    Wa = env_rng.standard_normal((D, A)) / np.sqrt(D)
    mine = list(range(rank, n_actors, nproc))
    state = {i: rng.standard_normal(D) for i in mine}
    ep = {i: 0 for i in mine}
    last = {i: deque() for i in mine}
    noise = {i: rng.uniform(-0.25, 0.25) for i in mine}            # one constant per actor (ppo_agent.py:60-61)
    zf = ZFilter(D)
    while True:
        msg = conn.recv()
        if msg == 'stop':
            break
        # fetch_parameter: rebuild the model from the published flat parameter vector
        off, layers = 0, []
        for l in range(3):
            k, m = dims[l], dims[l + 1]
            W = torch.from_numpy(par[off:off + k * m].reshape(m, k).copy()); off += k * m
            b = torch.from_numpy(par[off:off + m].copy()); off += m
            layers.append((W, b))
        log_var = torch.from_numpy(par[off:off + A].copy()).view(1, A); off += A
        zf.load(par[off:off + D].copy(), par[off + D:off + 2 * D].copy(), par[off + 2 * D:off + 2 * D + 1].copy())
        steps = 0
        for i in mine:
            s, dq = state[i], last[i]
            for _ in range(horizon):
                a, pdv = ppo_act(s.astype(np.float32), layers, log_var, zf, noise[i], eps=rng.standard_normal(A))
                s2 = np.tanh(Ws @ s + Wa @ a) + 0.01 * rng.standard_normal(D)
                r = -float(s @ s) / D + 0.1 * rng.standard_normal()
                ep[i] += 1
                done = ep[i] >= EPISODE_LEN
                dq.append((s.astype(np.float32), a, r, done, pdv))
                steps += 1
                if len(dq) == n:                                   # window complete: ship it, pop `stride` (= n) items
                    w_obs[i] = np.stack([e[0] for e in dq])
                    w_next[i, 0] = s2.astype(np.float32)
                    w_act[i] = np.stack([e[1] for e in dq])
                    w_rew[i] = [e[2] for e in dq]
                    w_done[i] = [float(e[3]) for e in dq]
                    w_pd[i] = np.stack([e[4] for e in dq])
                    dq.clear()
                if done:
                    dq.clear()
                    ep[i] = 0
                    s2 = rng.standard_normal(D)
                s = s2
            state[i] = s
        conn.send(steps)


class CpuSurreal:
    """Single-box Surreal on the host cores, restated by the oracle: P persistent actor processes (1024 logical actors
    spread over them), an in-process FIFO (oracle.replay.FIFO), np.stack aggregation (oracle.aggregator) and the torch-CPU
    learner (oracle.ppo.OraclePPOLearner).  One step() = every actor advances HORIZON env steps (1024 windows into the
    FIFO) while the learner consumes the previous step's 1024 windows and publishes -- actors and learner overlap with a
    one-step policy lag, like the GPU engine and like Surreal's asynchronous processes."""

    def __init__(self, n_actors=N_ACTORS, horizon=HORIZON, procs=None):
        import multiprocessing as mp
        import numpy as np
        import torch
        from multiprocessing import shared_memory
        from oracle.ppo import OraclePPOLearner
        from oracle.filters import ZFilter
        from oracle.replay import FIFO
        self.np, self.torch = np, torch
        self.n_actors, self.horizon = n_actors, horizon
        cores = os.cpu_count() or 1
        self.cores = cores
        self.procs = procs or max(1, min(64, cores - min(16, cores // 4)))
        D, A, n = OBS_DIM, ACT_DIM, horizon
        g = torch.Generator().manual_seed(0)
        da, dc = [D] + list(HIDDEN) + [A], [D] + list(HIDDEN) + [1]
        self.dims = da
        self.learner = OraclePPOLearner(_ref_layers(da, g), torch.zeros(1, A) - 1.0, _ref_layers(dc, g), ZFilter(D), A, n,
                                        n_actors, ppo_mode='clip', exp_interval=n_actors)
        self.fifo = FIFO(2 * n_actors, n_actors)
        n_par = sum(da[i] * da[i + 1] + da[i + 1] for i in range(3)) + A + 2 * D + 1
        shapes = dict(params=(n_par, 4), obs=(n_actors * n * D, 4), obs_next=(n_actors * D, 4), actions=(n_actors * n * A, 8),
                      rewards=(n_actors * n, 8), dones=(n_actors * n, 4), pd=(n_actors * n * 2 * A, 4))
        self.shms = {k: shared_memory.SharedMemory(create=True, size=c * s) for k, (c, s) in shapes.items()}
        self.par = np.ndarray((n_par,), dtype=np.float32, buffer=self.shms['params'].buf)
        self.w = dict(obs=np.ndarray((n_actors, n, D), dtype=np.float32, buffer=self.shms['obs'].buf),
                      obs_next=np.ndarray((n_actors, 1, D), dtype=np.float32, buffer=self.shms['obs_next'].buf),
                      actions=np.ndarray((n_actors, n, A), dtype=np.float64, buffer=self.shms['actions'].buf),
                      rewards=np.ndarray((n_actors, n), dtype=np.float64, buffer=self.shms['rewards'].buf),
                      dones=np.ndarray((n_actors, n), dtype=np.float32, buffer=self.shms['dones'].buf),
                      pd=np.ndarray((n_actors, n, 2 * A), dtype=np.float32, buffer=self.shms['pd'].buf))
        self._publish()
        ctx = mp.get_context('spawn')
        self.conns, self.ps = [], []
        names = {k: v.name for k, v in self.shms.items()}
        for r in range(self.procs):
            a, b = ctx.Pipe()
            p = ctx.Process(target=_ref_actor_proc, args=(r, self.procs, b, names, n_actors, horizon), daemon=True)
            p.start()
            self.conns.append(a)
            self.ps.append(p)
        self.threads = None
        self.pending = False
        self.learn_s, self.actor_s = [], []

    def _publish(self):
        """ParameterPublisher.publish (parameter_server.py:20-80): flat state vector into shared memory."""
        L, np, off = self.learner, self.np, 0
        for (W, b) in L.actor:
            k = W.numel()
            self.par[off:off + k] = W.detach().numpy().reshape(-1); off += k
            self.par[off:off + b.numel()] = b.detach().numpy(); off += b.numel()
        A, D = ACT_DIM, OBS_DIM
        self.par[off:off + A] = L.log_var.detach().numpy().reshape(-1); off += A
        self.par[off:off + D] = L.zf.running_sum.numpy(); self.par[off + D:off + 2 * D] = L.zf.running_sumsq.numpy()
        self.par[off + 2 * D] = float(L.zf.count)

    def _go(self):
        self._t_go = time.time()
        for c in self.conns:
            c.send('go')
        self.pending = True

    def _collect(self):
        """Wait for the actors, then insert their windows one by one (replay/base.py insert) in actor order."""
        n = sum(c.recv() for c in self.conns)
        self.actor_s.append(time.time() - self._t_go)
        self.pending = False
        w = {k: v.copy() for k, v in self.w.items()}
        for i in range(self.n_actors):
            self.fifo.insert({k: v[i] for k, v in w.items()})
        return n

    def _learn(self):
        from oracle.aggregator import multistep_aggregate
        np = self.np
        wins = self.fifo.sample(self.n_actors)
        t0 = time.time()
        batch = multistep_aggregate([dict(obs=x['obs'], obs_next=x['obs_next'][0], actions=x['actions'], rewards=x['rewards'],
                                          dones=x['dones'], pd=x['pd']) for x in wins])
        st = self.learner.learn(batch)
        self.learner.publish_parameter()
        self._publish()
        self.learn_s.append(time.time() - t0)
        return st

    def prime(self):
        """Fill the FIFO with the first 1024 windows and pick the learner's thread count once (torch-CPU does not scale
        to every core on these small GEMMs)."""
        torch = self.torch
        self._go()
        self._collect()
        best = None
        snapshot = self.fifo.q.copy()
        for nt in [t for t in (8, 16, 32) if t <= max(8, self.cores)]:
            torch.set_num_threads(nt)
            self.fifo.q = snapshot.copy()
            t0 = time.time()
            self._learn()
            dt = time.time() - t0
            if best is None or dt < best[0]:
                best = (dt, nt)
        self.threads = best[1]
        torch.set_num_threads(self.threads)
        self.fifo.q = snapshot.copy()
        self.learn_s = []

    def step(self):
        """Actors produce windows k+1 while the learner trains on windows k; returns env steps taken."""
        self._go()
        self._learn()
        return self._collect()

    def close(self):
        for c in self.conns:
            try:
                c.send('stop')
            except Exception:
                pass
        for p in self.ps:
            p.join(timeout=5)
            if p.is_alive():
                p.kill()
        for s in self.shms.values():
            s.close()
            s.unlink()


def cpu_reference(steps=3, warmup=1):
    """`warmup + steps` real steps of the CPU engine; env-steps/s over the timed steps (wall clock)."""
    eng = CpuSurreal()
    try:
        eng.prime()
        for _ in range(warmup):
            eng.step()
        eng.learn_s, eng.actor_s = [], []
        t0 = time.time()
        n = 0
        for _ in range(steps):
            n += eng.step()
        dt = time.time() - t0
        med = lambda v: sorted(v)[len(v) // 2] if v else None  # noqa: E731
        return {'value': n / dt, 'unit': 'env-steps/s', 'cores': eng.procs + eng.threads, 'host_cores': eng.cores,
                'kind': 'port', 'actor_processes': eng.procs, 'learner_threads': eng.threads, 'steps': steps, 'warmup': warmup,
                'seconds': dt, 'ms_per_step': dt / steps * 1e3, 'actors_phase_s': med(eng.actor_s),
                'learner_learn_s': med(eng.learn_s),
                'actors_only_steps_per_s': (N_ACTORS * HORIZON / med(eng.actor_s)) if eng.actor_s else None,
                'learner_updates_per_s': steps / dt,
                'sample': '%d measured full steps (after %d warm-up): %d persistent actor processes run 1024 logical actors x %d '
                          'env steps (batch-1 torch forward + numpy sampling + deque windowing) -> shared-memory windows -> '
                          'FIFO -> np.stack aggregation -> oracle PPO learn() on %d torch threads -> publish; actors overlap '
                          'the learner (one-step lag); ZeroMQ/pyarrow hops omitted' % (steps, warmup, eng.procs, HORIZON,
                                                                                      eng.threads)}
    finally:
        eng.close()


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    r = cpu_reference(steps=args.steps, warmup=args.warmup)
    value = r['value']
    out = {'impl': 'reference', 'metric': 'env-steps/sec', 'value': value, 'unit': 'env-steps/s',
           'n_gpus': int(os.environ.get('WORLD_SIZE', args.gpus)), 'steps': args.steps, 'warmup': args.warmup,
           'ms_per_step': r['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
           'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
           'config': bench_config(int(os.environ.get('WORLD_SIZE', args.gpus))),
           'engine': 'cpu: %d actor processes + %d learner threads, actors overlap the learner' % (r['actor_processes'],
                                                                                                 r['learner_threads']),
           'learner_updates_per_sec': r['learner_updates_per_s'], 'cpu_baseline': r,
           'e2e': {'value': value, 'unit': 'env-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(out))


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', type=str, default='ours', choices=['ours', 'reference'])
    ap.add_argument('--sequential', action='store_true', help='rollout then learn on one stream (no actor/learner overlap)')
    ap.add_argument('--lite', action='store_true', help='skip the e2e and CPU-baseline legs (profiling runs under ncu)')
    ap.add_argument('--workload', type=str, default='cfg2', choices=['cfg2', 'cfg5'],
                    help='cfg2: BASELINE configs[1] (the metric; weak scaling).  cfg5: configs[4], 4096 actors x horizon 256 in total, '
                         'sharded over the ranks (strong scaling; use with --lite)')
    ap.add_argument('--dump-outputs', type=str, default=None, metavar='DIR',
                    help='after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and a.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of --impl ours')
    if a.workload == 'cfg5':
        WORKLOAD = 'cfg5'
        N_ACTORS, HORIZON = 4096 // int(os.environ.get('WORLD_SIZE', 1)), 256
        EPISODE_LEN = 512
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)
