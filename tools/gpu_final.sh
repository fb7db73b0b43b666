#!/bin/bash
# round-2 evidence pass on ONE B200: tests, benches, profiles (outputs: gpurun_out/r02_*)
mkdir -p gpurun_out
O=gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > $O/r02_gpu.txt 2>&1
timeout 1800 python -m pytest tests -q -m gpu > $O/r02_pytest_gpu.txt 2>&1; echo "rc=$?" >> $O/r02_pytest_gpu.txt
timeout 300 python __graft_entry__.py smoke > $O/r02_smoke.txt 2>&1
LFR_BENCH_DEBUG=1 timeout 600 python bench.py --steps 20 --warmup 3 > $O/r02_bench_cfg2.json 2> $O/r02_bench_cfg2.err
timeout 600 python bench.py --impl reference --steps 20 --warmup 3 > $O/r02_bench_cfg2_reference.json 2> $O/r02_bench_cfg2_reference.err
timeout 600 python bench.py --steps 10 --warmup 3 --workload cfg3 > $O/r02_bench_cfg3.json 2> $O/r02_bench_cfg3.err
timeout 600 python bench.py --steps 10 --warmup 3 --workload cfg4 > $O/r02_bench_cfg4.json 2> $O/r02_bench_cfg4.err
timeout 300 python tools/gpu_cycles.py cfg2 > $O/r02_cycles_cfg2.txt 2>&1
timeout 300 python tools/gpu_zc_timeline.py cfg2 0 > $O/r02_timeline_zero_copy.txt 2>&1
timeout 300 python tools/gpu_zc_timeline.py cfg2 8 > $O/r02_timeline_hbm.txt 2>&1
timeout 600 python tools/gpu_batched.py > $O/r02_batched.txt 2>&1
timeout 600 python tools/gpu_e2e_timeline.py cfg2 > $O/r02_e2e_cfg2.txt 2>&1
timeout 600 python tools/gpu_e2e_timeline.py cfg5 > $O/r02_e2e_cfg5.txt 2>&1
timeout 900 python tools/gpu_cfg5.py cfg5 > $O/r02_cfg5_madrid_scale_1gpu.json 2> $O/r02_cfg5.err
timeout 900 python tools/gpu_cta_parity.py > $O/r02_cta_parity.txt 2>&1
timeout 600 python tools/gpu_tier_timeline.py cfg4 > $O/r02_tier_timeline_cfg4.txt 2>&1
timeout 600 python tools/gpu_cfg5_timeline.py cfg5 1 > $O/r02_cta_timeline_cfg5.txt 2>&1
timeout 900 compute-sanitizer --tool memcheck python tools/gpu_sanitize.py > $O/r02_sanitizer.txt 2>&1
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $O/r02_ncu_launches_bench_cfg2.csv python bench.py --steps 2 --warmup 3 > $O/r02_bench_under_ncu.log 2>&1
timeout 900 ncu --set full --clock-control none --import-source on -k regex:solve_ -c 11 -o $O/r02_full python tools/gpu_prof.py cfg2 1 > $O/r02_ncu_full.log 2>&1
ncu -i $O/r02_full.ncu-rep --page raw --csv > $O/r02_full_raw.csv 2>/dev/null
timeout 1500 ncu --set full --clock-control none --import-source on -k regex:solve_cta_kernel -c 3 -o $O/r02_cta_full python tools/gpu_cfg5.py cfg5 > $O/r02_ncu_cta.log 2>&1
ncu -i $O/r02_cta_full.ncu-rep --page raw --csv > $O/r02_cta_full_raw.csv 2>/dev/null
ncu -i $O/r02_cta_full.ncu-rep --page details > $O/r02_cta_full_details.txt 2>/dev/null
rm -f $O/r02_cta_full.ncu-rep
tail -n 3 $O/r02_pytest_gpu.txt; tail -n 2 $O/r02_smoke.txt
head -12 $O/r02_cycles_cfg2.txt; cat $O/r02_e2e_cfg2.txt $O/r02_e2e_cfg5.txt; grep -E "solve_ms|host_stage_s|plan_create_s" $O/r02_cfg5_madrid_scale_1gpu.json; tail -n 4 $O/r02_sanitizer.txt
python - <<'PY'
import json,glob
for f in sorted(glob.glob('gpurun_out/r02_bench_*.json')):
    try:
        d=json.loads(open(f).read().strip().splitlines()[-1])
        print(f, 'ms/step %.4f'%d['ms_per_step'], 'value %.3g'%d['value'], 'e2e', d['e2e'].get('ms_per_step'), d['e2e'].get('stages_ms'), 'frac', (d.get('roofline') or {}).get('frac'), 'cpu', d['cpu_baseline'].get('ms_per_step'), d.get('total_scope',{}).get('host_stage_ms'))
    except Exception as e:
        print(f,'ERR',e)
PY
