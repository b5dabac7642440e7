#!/bin/bash
# exact tcgen05 engine (round-2 structure), and an A/B of the round-1 tree (_ab_r01, commit 9401463) against
# the current one on the SAME box (default workload and the logging workload)
set -u
O=gpurun_out
P=/tmp/ctk_prof
mkdir -p $O $P
timeout 900 python -m pytest tests -m gpu -q --timeout 600 -k "tcgen05 or mlp or top_m" 2>&1 | tail -15 | tee $O/pytest_gpu_mlp.txt
python bench.py --workload mppi_mlp_c4 --mlp-engine tcgen05 --steps 10 --warmup 3 > $O/bench_mlp_exact_v2.json 2> $O/bench_mlp_exact_v2.err
for i in 1 2; do
  (cd _ab_r01 && python bench.py > ../$O/ab_r01_default_$i.json 2> ../$O/ab_r01_default_$i.err)
  python bench.py > $O/ab_r02_default_$i.json 2> $O/ab_r02_default_$i.err
done
CTK_K1_FINISHER_SHARE=1.0 python bench.py > $O/ab_r02_default_share1.json 2> $O/ab_r02_default_share1.err
(cd _ab_r01 && python bench.py --workload mppi_ode_1m_log > ../$O/ab_r01_log.json 2> ../$O/ab_r01_log.err)
python bench.py --workload mppi_ode_1m_log > $O/ab_r02_log.json 2> $O/ab_r02_log.err
timeout 600 ncu --set full --clock-control none --import-source on -k regex:mppi_rollout_kernel -s 4 -c 1 -o $P/prof_mlp_tc_r02_exact_v2 -f python bench.py --workload mppi_mlp_c4 --mlp-engine tcgen05 --steps 3 --warmup 3 > $O/ncu_mlp_exact_v2.log 2>&1
python tools/ncu_summary.py $P/prof_mlp_tc_r02_exact_v2.ncu-rep > $O/prof_mlp_tc_r02_exact_v2_summary.txt 2>&1
for f in $O/bench_mlp_exact_v*.json $O/ab_*.json; do echo $f; python -c "
import json,sys
d=json.loads(open('$f').read().strip().splitlines()[-1]); r=d.get('roofline') or {}
print('  ms/step', d['ms_per_step'], 'kernel_ms', r.get('kernel_ms'), 'frac', r.get('frac'), 'pipelined', (d.get('pipelined') or {}).get('ms_per_step'))
"; done
echo done
