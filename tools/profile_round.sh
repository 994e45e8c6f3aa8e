#!/bin/bash
# Reproduces the files under profiles/ (run on a B200 box from the repo root, e.g. through gpurun).
# Every ncu pass follows a plain run of the same command that exited 0; reports are summarised on the box by
# tools/summarize_ncu.py and the .ncu-rep files deleted (they are tens of MB each).
set +e
O=${1:-gpurun_out}
TAG=${2:-r2}
mkdir -p $O
CMD="python bench.py --nt 300 --steps 1 --warmup 3 --no-cpu-baseline --no-track-a --no-extras --no-configs"

# 1. launch list of the bench command (kernel share of the step)
$CMD > $O/plain_a.log 2>&1 && ncu --metrics gpu__time_duration.sum --clock-control none -c 12000 --csv \
    --log-file $O/launches.csv $CMD > $O/ncu_a.log 2>&1
python tools/summarize_ncu.py launches $O/launches.csv > $O/${TAG}_launches_bench_nt300.txt; rm -f $O/launches.csv

# 2. the dominant kernel, cold caches (ncu default) and warm caches (--cache-control none).  The bench first models the
#    observed data of its 4 shots (4 x 300 plain forward launches), then runs the gradients: -s 1496 -c 8 takes the last four
#    forward-save launches of the first gradient and the first four adjoint launches (propagate-only / deferred-imaging pairs).
for mode in cold warm; do
    extra=""; [ $mode = warm ] && extra="--cache-control none"
    $CMD > $O/plain_b.log 2>&1 && ncu --set full $extra --clock-control none --import-source on -k regex:fd2d_step \
        -s 1496 -c 8 -o $O/prof_fd2d_$mode $CMD > $O/ncu_b_$mode.log 2>&1
    ncu -i $O/prof_fd2d_$mode.ncu-rep --page raw --csv > /tmp/p.csv 2>/dev/null
    python tools/summarize_ncu.py raw /tmp/p.csv > $O/${TAG}_fd2d_step_ncu_full_$mode.txt; rm -f $O/prof_fd2d_$mode.ncu-rep
done
# 3. 3-D kernel (single GPU, 384^3)
python tools/step_bench3d.py 384 20 > $O/${TAG}_fd3d_bench.txt 2>&1 && ncu --set full --clock-control none -k regex:fd3d_step \
    -s 30 -c 2 -o $O/prof_fd3d python tools/step_bench3d.py 384 20 > $O/ncu_d.log 2>&1
ncu -i $O/prof_fd3d.ncu-rep --page raw --csv > /tmp/p.csv 2>/dev/null
python tools/summarize_ncu.py raw /tmp/p.csv > $O/${TAG}_fd3d_step_ncu_full.txt; rm -f $O/prof_fd3d.ncu-rep

# 4. Track A likelihood kernel
python tools/mc_bench.py 2000000 > $O/${TAG}_mc_bench.txt 2>&1 && ncu --set full --clock-control none -k regex:mc_eval \
    -s 2 -c 1 -o $O/prof_mc python tools/mc_bench.py 2000000 > $O/ncu_e.log 2>&1
ncu -i $O/prof_mc.ncu-rep --page raw --csv > /tmp/p.csv 2>/dev/null
python tools/summarize_ncu.py raw /tmp/p.csv > $O/${TAG}_mc_eval_ncu_full.txt; rm -f $O/prof_mc.ncu-rep

# 5. Track A tensor-core likelihood kernel (default path): the first evaluation of tools/mc_bench.py at N = 4e6
python tools/mc_bench.py 4000000 > $O/plain_u.log 2>&1 && ncu --set full --clock-control none --import-source on -k regex:mc_umma_kernel \
    -c 1 -o $O/prof_umma python tools/mc_bench.py 4000000 > $O/ncu_umma.log 2>&1
ncu -i $O/prof_umma.ncu-rep --page raw --csv > /tmp/p.csv 2>/dev/null
python tools/summarize_ncu.py raw /tmp/p.csv > $O/${TAG}_mc_umma_ncu_full.txt; rm -f $O/prof_umma.ncu-rep
du -sh $O
