#!/bin/bash
# Round-2 evidence on ONE GPU: parity suite, smoke, bench lines of every config (both arms of cfg2), ncu launch lists and full
# captures of the kernels of a cfg2 step plus the draw kernel at cfg3 / cfg5, compute-sanitizer.
# usage: tools/gpu_round2.sh <tag>   (outputs under gpurun_out/<tag>_*; summarise with tools/ncu_summary.py)
TAG=${1:-r2x}
O=gpurun_out
mkdir -p $O
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > $O/${TAG}_smi.txt 2>&1
timeout 1500 python -m pytest tests -m gpu -x -q > $O/${TAG}_pytest.log 2>&1; echo "pytest rc=$?" | tee -a $O/${TAG}_pytest.log
tail -3 $O/${TAG}_pytest.log
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $O/${TAG}_smoke.log 2>&1; echo "smoke rc=$?"; tail -1 $O/${TAG}_smoke.log
timeout 900 python bench.py > $O/${TAG}_bench_default.json 2> $O/${TAG}_bench_default.err; echo "bench (driver's command) rc=$?"
timeout 900 python bench.py --steps 500 --warmup 10 --no-sharded > $O/${TAG}_bench_cfg2.json 2> $O/${TAG}_bench_cfg2.err; echo "bench cfg2 500 steps rc=$?"
timeout 600 python bench.py --impl reference --steps 40 --warmup 5 > $O/${TAG}_bench_cfg2_reference.json 2> $O/${TAG}_bench_ref.err; echo "ref rc=$?"
timeout 600 python bench.py --streaming --no-cpu-baseline --no-sharded > $O/${TAG}_bench_cfg2_streaming.json 2> $O/${TAG}_bench_streaming.err; echo "streaming rc=$?"
for wl in cfg1 cfg3 cfg4 cfg5; do
  timeout 900 python bench.py --workload $wl --steps 100 --warmup 10 > $O/${TAG}_bench_$wl.json 2> $O/${TAG}_bench_$wl.err; echo "$wl rc=$?"
done
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $O/${TAG}_launches_cfg2.csv python bench.py --steps 20 --warmup 3 --no-cpu-baseline --no-sharded > $O/${TAG}_ncu_launch.log 2>&1; echo "ncu launches cfg2 rc=$?"
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 60 --csv --log-file $O/${TAG}_launches_cfg3.csv python bench.py --workload cfg3 --steps 5 --warmup 3 --no-cpu-baseline > /dev/null 2>&1; echo "ncu launches cfg3 rc=$?"
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 60 --csv --log-file $O/${TAG}_launches_cfg5.csv python bench.py --workload cfg5 --steps 3 --warmup 3 --no-cpu-baseline --no-sharded > /dev/null 2>&1; echo "ncu launches cfg5 rc=$?"
for K in cs_search2 cs_sort cs_wedge; do
  timeout 600 ncu --set full --clock-control none --import-source on -k regex:${K}_kernel -s 30 -c 1 -f -o $O/${TAG}_${K#cs_}_cfg2 python bench.py --steps 20 --warmup 3 --no-cpu-baseline --no-sharded > $O/${TAG}_ncu_${K#cs_}.log 2>&1; echo "ncu $K rc=$?"
done
timeout 600 ncu --set full --clock-control none --import-source on -k regex:cs_wedge -s 4 -c 1 -f -o $O/${TAG}_wedge_cfg3 python bench.py --workload cfg3 --steps 3 --warmup 3 --no-cpu-baseline > $O/${TAG}_ncu_wedge_cfg3.log 2>&1; echo "ncu wedge cfg3 rc=$?"
timeout 600 ncu --set full --clock-control none --import-source on -k regex:cs_wedge -s 7 -c 1 -f -o $O/${TAG}_wedge_cfg5 python bench.py --workload cfg5 --steps 3 --warmup 3 --no-cpu-baseline --no-sharded > $O/${TAG}_ncu_wedge_cfg5.log 2>&1; echo "ncu wedge cfg5 rc=$?"
bash tools/sanitize.sh $TAG > $O/${TAG}_sanitize.out 2>&1; grep -c "0 errors\|0 hazards" $O/${TAG}_sanitize.out
ls $O | grep "^${TAG}_" | wc -l
