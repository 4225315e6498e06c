#!/bin/bash
# Run on the GPU box (gpurun): launch list of one bench step + full ncu captures of the dominant kernels.
# Outputs land in gpurun_out/ ; summaries are written into profiles/ by tools/summarize_profiles.py (run here).
mkdir -p gpurun_out
# eager launches so that every kernel is a separate ncu record (graphs replay the same sequence)
SB200_CUDA_GRAPH=0 timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 4000 --csv \
    --log-file gpurun_out/launches.csv python bench.py --steps 1 --warmup 3 --lite --sequential > gpurun_out/launches_bench.log 2>&1
echo "launch list rc=$?"
timeout 600 ncu --set full --clock-control none --import-source on -k ppo_rollout2_kernel -s 2 -c 1 \
    -o gpurun_out/prof_rollout -f python tools/prof_rollout.py 128 1 > gpurun_out/prof_rollout.log 2>&1
echo "rollout capture rc=$?"
timeout 300 ncu --set full --clock-control none --import-source on -k regex:mlp3_tc5 -s 2 -c 1 -f -o gpurun_out/prof_tc5 \
    tools/tc5_harness prof > gpurun_out/prof_tc5.log 2>&1
echo "tc5 capture rc=$?"
ls -la gpurun_out | head -40
# round 2b: the one-launch learner kernel, the v2 rollout kernel (matched by the ppo_rollout regex above), GAE at 2^18 windows
timeout 300 ncu --set full --clock-control none --import-source on -k regex:ppo_epochs2 -s 2 -c 1 -f -o gpurun_out/prof_epochs2 \
    python tools/prof_epoch2.py > gpurun_out/prof_epochs2.log 2>&1
echo "epochs2 capture rc=$?"
timeout 300 ncu --set full --clock-control none --import-source on -k regex:gae_full -s 2 -c 1 -f -o gpurun_out/prof_gae_large \
    python tools/prof_gae.py > gpurun_out/prof_gae_large.log 2>&1
echo "gae capture rc=$?"
