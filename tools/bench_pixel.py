#!/usr/bin/env python
"""BASELINE configs[3]: PPO on synthetic pixel observations (uint8 84x84x4), 256 actors, CNN encoder, horizon 128.

Not the bench.py headline (that is configs[1]); a tracked measurement for DESIGN.md.  One step = 128 env steps of all 256
actors (CNN stem + actor head + sampling + device pixel env + window staging of uint8 frames into the HBM FIFO, one CUDA
graph per chunk) followed by PPOLearner.learn() on the 256 windows (stem + critic over 33 024 frames, GAE, 10 + 10 epochs
that train the shared stem through both optimisers).  Under torchrun every rank runs its own 256 actors (weak scaling) and
the learner is data-parallel.

``--low-dim D`` adds a D-float low-dim input next to the frame (mixed observations, the robosuite spec of
ppo_configs.py:111-114): the records carry frame + low-dim, the heads take cat(zfilter(low_dim), features) and the z-filter
is on.  Single GPU only (the mixed learner has no data-parallel path).

    python tools/bench_pixel.py [steps] [--low-dim D]   |   torchrun --nproc-per-node N tools/bench_pixel.py [steps]
"""
import copy
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402


def main():
    import argparse
    import torch.distributed as dist
    ap = argparse.ArgumentParser()
    ap.add_argument('steps', type=int, nargs='?', default=5)
    ap.add_argument('--low-dim', type=int, default=0, help='floats of low-dim input next to the frame (0: pixel only)')
    args = ap.parse_args()
    steps, Dl = args.steps, args.low_dim
    rank, world, local = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1)), int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('NCCL_MAX_NCHANNELS', '4')
        dist.init_process_group('nccl', device_id=dev)
    from surreal_b200.session import Config
    from surreal_b200.main.ppo_configs import (PPO_DEFAULT_LEARNER_CONFIG, PPO_DEFAULT_ENV_CONFIG, PPO_DEFAULT_SESSION_CONFIG,
                                               make_synthetic_pixel_env_config)
    from surreal_b200.launch import SurrealDefaultLauncher
    from surreal_b200.agent import PPOAgent
    from surreal_b200.learner import PPOLearner
    from surreal_b200.replay import FIFOReplay
    N, T, SHAPE, A = 256, 128, (4, 84, 84), 8
    lc = Config(copy.deepcopy(PPO_DEFAULT_LEARNER_CONFIG.to_dict()))
    ec = Config(copy.deepcopy(PPO_DEFAULT_ENV_CONFIG.to_dict()))
    sc = Config(copy.deepcopy(PPO_DEFAULT_SESSION_CONFIG.to_dict()))
    sc.folder = tempfile.mkdtemp(prefix='sb200_pixel_')
    lc.model.actor_fc_hidden_sizes, lc.model.critic_fc_hidden_sizes, lc.model.cnn_feature_dim = [256, 256], [256, 256], 256
    lc.algo.ppo_mode, lc.algo.rnn.if_rnn_policy, lc.algo.use_z_filter = 'clip', False, False
    lc.algo.n_step = lc.algo.stride = T
    lc.replay.batch_size, lc.replay.memory_size = N, 2 * N
    lc.parameter_publish.exp_interval, lc.parameter_publish.min_publish_interval = N, 0.0
    make_synthetic_pixel_env_config(ec, N, SHAPE, A, seed=rank)
    if Dl > 0:
        if world > 1:
            raise SystemExit('--low-dim: the mixed-observation learner runs on one GPU')
        ec.obs_spec = {'low_dim': {'robot-state': (Dl,)}, 'pixel': {'camera0': SHAPE}}
        lc.algo.use_z_filter = True
    ec.limit_episode_length = 2 * T
    sc.agent.fetch_parameter_interval = T
    la = SurrealDefaultLauncher(PPOAgent, PPOLearner, FIFOReplay, sc, ec, lc)
    agent, replay, learner = la.setup_engine()
    if world > 1:
        learner.enable_data_parallel(dist.group.WORLD)

    def step():
        agent.main_loop(max_steps=T)
        learner.main_loop()
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * steps + 1)]
    ev[0].record()
    for i in range(steps):
        agent.main_loop(max_steps=T)
        ev[2 * i + 1].record()
        learner.main_loop()
        ev[2 * i + 2].record()
    torch.cuda.synchronize()
    roll = sorted(ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(steps))[steps // 2]
    learn = sorted(ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(steps))[steps // 2]
    total = ev[0].elapsed_time(ev[-1])
    if world > 1:
        t = torch.tensor([total], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total = float(t.item())
    if rank == 0:
        frame = SHAPE[0] * SHAPE[1] * SHAPE[2]
        mixed = ' + %d low-dim floats (z-filtered)' % Dl if Dl else ''
        print(json.dumps({'workload': 'PPO synthetic pixel 84x84x4 uint8%s, 256 actors per GPU x horizon 128, CNN 16k8s4-32k4s2-FC256 + '
                                      '2x256 heads (BASELINE configs[3])' % mixed, 'low_dim': Dl, 'n_gpus': world, 'steps': steps,
                          'gpu': torch.cuda.get_device_name(dev),
                          'env_steps_per_s': N * T * steps * world / (total / 1e3), 'ms_per_step': total / steps,
                          'rollout_ms': roll, 'learn_ms': learn, 'frame_bytes_in_hbm': frame, 'algorithmic_frame_bytes': 28224,
                          'frames_through_stem_per_step': N * T + N * (T + 1) + 21 * N * 3,
                          'stem_flop_per_frame': 5.93e6}))
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        os._exit(0)


if __name__ == '__main__':
    main()
