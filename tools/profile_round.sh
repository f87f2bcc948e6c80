#!/bin/bash
# Round profile capture (run on the GPU box through gpurun): bench lines without a profiler first, then the ncu launch
# list of the same command, then one `--set full` capture of the top kernels.  Everything lands in gpurun_out/.
set -u
R=${1:-r2}
O=gpurun_out
mkdir -p $O
python bench.py > $O/${R}_bench_all.json 2> $O/${R}_bench_all.err || exit 1
python bench.py --impl reference --steps 2 --warmup 1 > $O/${R}_bench_reference.json 2> $O/${R}_bench_reference.err
python tools/stage_profile.py > $O/${R}_stage_profile.log 2>&1
python tools/nms_profile.py > $O/${R}_nms_phases.log 2>&1
python tools/msroialign_profile.py > $O/${R}_msroialign.log 2>&1
{ python tools/roi_bwd_probe.py; python tools/roi_bwd_probe.py cfg4; } > $O/${R}_roi_bwd_probe.log 2>&1
ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $O/${R}_bench_launches.csv \
    python bench.py --workload rpn --steps 3 --warmup 3 --no-cpu > $O/ncu1.log 2>&1
# (the launch geometry of the timed path: one NMS CTA per image, as region.ProposalPipeline runs it)
ncu --set full --clock-control none --import-source on -k regex:"nms_bucket|rpn_decode|topk_bucket" -s 12 -c 3 \
    -o $O/prof_${R}_proposal -f python bench.py --workload rpn --single-stream --nms-cluster 1 --steps 3 --warmup 3 --no-cpu > $O/ncu2.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:"roi_|sample_|region_loss" -c 8 \
    -o $O/prof_${R}_roi -f python tools/roi_one.py > $O/ncu3.log 2>&1
ls -la $O
