#!/bin/bash
# One GPU-box call that produces everything a round's profiles/ entry needs.
#   gpurun --timeout 900 -- 'bash tools/profile_round.sh r01e'
# Outputs land in gpurun_out/<tag>_*; copy the summaries you want judged into profiles/.
TAG=${1:-rXX}
LPS=${LPS:-11}     # kernel launches per 64-clip step on the default path (frontend, seg_table, conv12, conv3..6, td_in, 2 x td_sa, pool_final)
OUT=gpurun_out
mkdir -p $OUT
BENCH_PROF="python bench.py --steps 2 --warmup 1 --warmup-seconds 0 --skip-cpu"
python -c "import torch" 2>/dev/null     # page the image in
timeout 600 python -m pytest tests -m gpu -x -q > $OUT/${TAG}_pytest.log 2>&1
echo "pytest exit $?"; tail -3 $OUT/${TAG}_pytest.log
# full capture of one step (LPS launches per step; the first step is skipped), raw page exported on the box; the
# per-launch DRAM traffic table the bench line quotes (profiles/roofline_traffic.json) is refreshed from it
timeout 600 ncu --set full --clock-control none --launch-skip $LPS -c $LPS -f -o $OUT/${TAG}_full \
    $BENCH_PROF > $OUT/${TAG}_ncu_full.log 2>&1
echo "ncu full exit $?"
ncu -i $OUT/${TAG}_full.ncu-rep --page raw --csv > $OUT/${TAG}_full_raw.csv 2>/dev/null
python tools/ncu_summary.py $OUT/${TAG}_full_raw.csv $TAG > $OUT/${TAG}_ncu_summary.txt 2>&1
cp profiles/${TAG}_ncu_full_one_step.csv profiles/roofline_traffic.json $OUT/ 2>/dev/null
timeout 600 python bench.py > $OUT/${TAG}_bench_n1.json 2> $OUT/${TAG}_bench.err
echo "bench exit $?"; cut -c1-300 $OUT/${TAG}_bench_n1.json
# launch list of the same command (cold-cache, serialised): one warm step skipped, two steps listed
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none --launch-skip $LPS -c $((2 * LPS)) --csv \
    --log-file $OUT/${TAG}_launches_bench_steps2.csv $BENCH_PROF > $OUT/${TAG}_ncu_launches.log 2>&1
echo "ncu launches exit $?"
timeout 150 python tools/bench_configs.py > $OUT/${TAG}_bench_configs.log 2>&1
echo "bench_configs exit $?"; mv $OUT/bench_configs.json $OUT/${TAG}_bench_configs.json 2>/dev/null
ls -la $OUT | head -30
