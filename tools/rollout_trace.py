#!/usr/bin/env python
"""clock64 timeline of the persistent rollout kernel: builds a -DRF_TRACE variant of the library under tools/_trace/
(never the shipped .so), runs one chunk at the bench shape and prints, per phase, the cycles cluster 0's CTAs spent.

    python tools/rollout_trace.py build      # here (nvcc only)
    python tools/rollout_trace.py            # on the GPU box
"""
import ctypes as C
import glob
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
OUT = os.path.join(ROOT, 'tools', '_trace')
LIB = os.path.join(OUT, 'libsurreal_b200_trace.so')
# (stamp id, phase that ends at it) in the order math warp 0 of a CTA passes them in one step; stamp 0 is the step top
PHASES = [(18, 'input tile wait'), (3, 'L1 fma + push'), (4, 'L1 mbarrier wait'), (5, 'L2 fma'), (6, 'L2 sync'),
          (7, 'L2 reduce + push'), (9, 'L2 wait + head slices'), (10, 'head sync'), (19, 'slice sums'),
          (20, 'mean/sample/stores'), (21, 'env finalize'), (11, 'bookkeeping'), (12, 'commit_actor'), (13, 'x0 push')]


def build():
    from surreal_b200 import build as B
    os.makedirs(OUT, exist_ok=True)
    procs = []
    for src in B._sources():
        obj = os.path.join(OUT, os.path.basename(src)[:-3] + '.o')
        procs.append((obj, subprocess.Popen([B.NVCC] + B.FLAGS + ['-DRF_TRACE', '-c', src, '-o', obj], stdout=subprocess.PIPE,
                                            stderr=subprocess.STDOUT, text=True)))
    objs = []
    for obj, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            sys.stderr.write(out)
            raise SystemExit(1)
        objs.append(obj)
    subprocess.check_call([B.NVCC, '-shared', '-o', LIB] + objs + ['-lcudart'])
    print(LIB)


def main():
    import numpy as np
    import torch
    from surreal_b200 import _lib
    _lib.LIB_PATH = LIB
    from helpers import ppo_configs
    from surreal_b200.agent import PPOAgent
    from surreal_b200.replay import FIFOReplay
    from surreal_b200.env import SyntheticEnv
    N, D, A, T = 1024, 64, 8, 128
    lc, ec, sc = ppo_configs(D=D, A=A, actor_h=(256, 256), critic_h=(256, 256), n_step=128, stride=128, B=N, memory_size=4 * N)
    ec.num_envs = N
    R = FIFOReplay(lc, ec, sc)  # noqa: F841
    ag = PPOAgent(lc, ec, sc, 0, 'training')
    env = SyntheticEnv(N, D, A, limit_episode_length=256, seed=0)
    ag.env = w = ag.prepare_env_agent(env)
    w.reset()
    for _ in range(3):
        ag.rollout_chunk(T)
    torch.cuda.synchronize()
    tr = np.zeros((4, 8, 32), dtype=np.int64)
    L = _lib.lib()
    L.sb200_debug_rf_trace.argtypes = [C.c_void_p]
    assert L.sb200_debug_rf_trace(tr.ctypes.data_as(C.c_void_p)) == 0
    for cta in range(4):
        print('CTA %d (cycles per phase, median over steps)' % cta)
        d = tr[cta]
        prev, total = 0, 0.0
        for i, name in PHASES:
            c = np.median(d[:, i] - d[:, prev])
            print('   %-24s %7.0f' % (name, c))
            total += c
            prev = i
        step = np.median(d[1:, 0] - d[:-1, 0])
        print('   %-24s %7.0f   (step period %0.f)' % ('sum', total, step))
        print('   env warp: starts %+.0f from step top, busy %.0f' % (np.median(d[:, 16] - d[:, 0]), np.median(d[:, 17] - d[:, 16])))


if __name__ == '__main__':
    if len(sys.argv) > 1 and sys.argv[1] == 'build':
        build()
    else:
        main()
